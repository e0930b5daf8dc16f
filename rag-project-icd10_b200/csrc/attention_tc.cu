// attention_tc.cu -- tensor-core self-attention for short sequences (S <= 128, head dim 64), sm_100a.
//
// Replaces BertSelfAttention inside SentenceTransformer.encode (reference call sites
// services/embedding_service.py:81,97-102,120):  ctx = softmax(Q K^T / 8 + mask) V  per (sequence, head).
//
// A work item is (token tile, head).  A token tile packs G = floor(128 / S) whole sequences into
// the 128 MMA rows (G * S <= 128 rows used); the block-diagonal + length mask keeps sequences
// apart.  Per item:
//   TMA      Q, K, V tiles [128 x 64] bf16 (one 128-byte-swizzled K block each) -> shared memory
//   MMA 1    S = Q K^T           tcgen05 SS, M=128 N=128 K=64, fp32 in TMEM (128 columns)
//   softmax  thread == TMEM lane == query row: tcgen05.ld, mask, max, exp2, row sum; the
//            un-normalised P goes back to TMEM as packed bf16 (64 columns) with tcgen05.st
//   MMA 2    O = P V             tcgen05 TS: A = P from TMEM, B = V read MN-major from the same
//            swizzled tile TMA wrote (no transpose pass), M=128 N=64 K=128, fp32 in TMEM
//   epilogue tcgen05.ld O, scale by 1 / row sum, bf16 into a 128-byte-swizzled staging box, one TMA store of
//            the G*S x 64 box to ctx (r01d: direct 16-byte stores, 32 lines per instruction, were a third of
//            the kernel: 0.42 ms with them, 0.27 ms without)
// Two softmax warpgroups work on alternate items.  Each owns one S region in TMEM (128 columns; P
// overwrites its first 64 once the row has been read) and two O regions (64 columns each), and runs
// one item ahead of itself: softmax(j) -> epilogue(j - 2) -> softmax(j + 2) ..., so the P V MMA of item j and
// the Q K^T MMA of item j + 2 (issued back to back: the tensor pipe executes them in order, which is what
// protects P) run while the warpgroup drains the previous O.  r01c had one TMEM set per item and the
// warpgroup idle across both MMA round trips: 49 % of DRAM peak.  A 4-slot shared-memory ring keeps the
// loads of three items in flight.
//
// Warp roles (320 threads): warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer,
// warps 2..5 / 6..9 softmax warpgroups 0 / 1 (TMEM lane quarter = warp % 4).
//
// Sequences of 129 .. 512 tokens (the token-classification path) run the SAME kernel in split-KV mode: a work item is
// (sequence, head, 128-query tile, 128-key tile); the softmax of an item is local to its key tile, the item stores its
// normalised partial output as bf16 into a [key tile][padded row][H] buffer plus (row max in the log2 domain, row
// sum) per (key tile, head, row), and attention_combine_kernel merges the <= 4 partials of a row with the weights
// exp2(m_t - m) sum_t -- the flash-decoding split, so no kernel keeps a running max across tiles.
//
// The hidden size H is a template parameter (768: 12 heads, 1024: 16 heads); it sets the qkv row stride 3H, the ctx
// row stride, the head count and the split-KV buffers.  Tiles, TMEM and shared memory are per head and do not change.
//
// Roofline: HBM (reads the 3H-wide qkv rows once, writes ctx once); the math is ~1 % of a layer.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "encoder_kernels.h"
#include "ptx.cuh"

namespace icd {
namespace {

constexpr int HD = 64;
constexpr int kTile = 128;
constexpr int kSlots = 4;
constexpr int kTileBytes = kTile * HD * 2;  // 16 KiB
constexpr int kSlotBytes = 3 * kTileBytes;  // Q, K, V
constexpr int kThreads = 320;
constexpr int kTmemCols = 512;
constexpr int kOBase = 256;    // TMEM columns: S/P of warpgroup 0 | S/P of warpgroup 1 | four O regions of 64
constexpr int kSmemBytes = kSlots * kSlotBytes + 2 * kTileBytes /*ctx staging, one box per warpgroup*/ + 1024 + 256;

struct AttParams {
  const int32_t* lens;
  int B, S, G, tiles;
  // split-KV mode (S > 128): QT = ceil(S / 128) query / key tiles per sequence, S_pad = QT * 128 rows per sequence in the
  // partial buffers, part_stats [QT][heads][B * S_pad] (log2-domain row max, row sum)
  int QT, S_pad;
  float2* part_stats;
#ifdef ICD_PROFILING
  int dbg;  // ICD_ATTN_DBG (profiling builds only): 1 = skip the ctx stores, 2 = every item loads tile 0 (L2 hits)
#endif
};

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int H>
__global__ void __launch_bounds__(kThreads, 1)
attention_tc_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_ctx,
                    const AttParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char* stage_o = smem + kSlots * kSlotBytes;  // [2 warpgroups][128 rows x 128 bytes], 1024-aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_o + 2 * kTileBytes);
  uint64_t* full_bar = bars;             // [4] TMA landed
  uint64_t* empty_bar = bars + 4;        // [4] P V of the item retired: slot reusable
  uint64_t* sfull_bar = bars + 8;        // [2] S ready in TMEM (per warpgroup)
  uint64_t* pready_bar = bars + 10;      // [2] P written by all 128 rows (per warpgroup)
  uint64_t* ofull_bar = bars + 12;       // [4] O ready in TMEM (per O region)
  uint64_t* ofree_bar = bars + 16;       // [4] O region drained by all 128 rows
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(bars + 20);
  constexpr int kHeads = H / HD;

  const int n_items = p.tiles * kHeads;
  const int n_local = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tmap(&tmap_qkv);
    ptx::prefetch_tmap(&tmap_ctx);
    for (int s = 0; s < kSlots; ++s) {
      ptx::mbar_init(ptx::smem_u32(&full_bar[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&empty_bar[s]), 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(ptx::smem_u32(&sfull_bar[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&pready_bar[s]), 128);
    }
    for (int s = 0; s < 4; ++s) {
      ptx::mbar_init(ptx::smem_u32(&ofull_bar[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&ofree_bar[s]), 128);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(ptx::smem_u32(tmem_holder), kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  // barriers and tensor memory are set up: let the next kernel of the forward start its own prologue, then wait for the
  // QKV projection to have completed before the first load
  ptx::griddep_launch();
  ptx::griddep_wait();

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      for (int j = 0; j < n_local; ++j) {
        const int item = (int)blockIdx.x + j * (int)gridDim.x;
        const int tile = item / kHeads, head = item % kHeads;
#ifdef ICD_PROFILING
        const int row0 = (p.dbg & 2) ? 0 : tile * p.G * p.S;
#else
        const int row0 = tile * p.G * p.S;
#endif
        int q_row0 = row0, k_row0 = row0;
        if (p.QT > 0) {  // split-KV: tile = (sequence, query tile, key tile)
          const int seq = tile / (p.QT * p.QT), qt = (tile / p.QT) % p.QT, kt = tile % p.QT;
          q_row0 = seq * p.S + qt * kTile;
          k_row0 = seq * p.S + kt * kTile;
        }
        const int slot = j % kSlots;
        ptx::mbar_wait(ptx::smem_u32(&empty_bar[slot]), ((j / kSlots) & 1) ^ 1);
        const uint32_t fb = ptx::smem_u32(&full_bar[slot]);
        ptx::mbar_expect_tx(fb, kSlotBytes);
        const uint32_t dst = ptx::smem_u32(smem + (size_t)slot * kSlotBytes);
        ptx::tma_load_2d(dst, &tmap_qkv, fb, head * HD, q_row0);
        ptx::tma_load_2d(dst + kTileBytes, &tmap_qkv, fb, H + head * HD, k_row0);
        ptx::tma_load_2d(dst + 2 * kTileBytes, &tmap_qkv, fb, 2 * H + head * HD, k_row0);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc_s = ptx::make_idesc_bf16(kTile, kTile);
      constexpr uint32_t idesc_o = ptx::make_idesc_bf16(kTile, HD) | (1u << 16);  // B (= V) is MN-major
      // item j: warpgroup w = j & 1, its i-th item (i = j >> 1); O region r = j & 3
      auto issue_s = [&](int j) {
        const int slot = j % kSlots, w = j & 1;
        ptx::mbar_wait(ptx::smem_u32(&full_bar[slot]), (j / kSlots) & 1);
        ptx::tc_fence_after();
        const uint32_t sq = ptx::smem_u32(smem + (size_t)slot * kSlotBytes);
        const uint32_t sk = sq + kTileBytes;
        const uint32_t d = tmem_base + (uint32_t)(w * kTile);
#pragma unroll
        for (int k4 = 0; k4 < HD / 16; ++k4)
          ptx::mma_ss(d, ptx::make_desc_k128(sq + k4 * 32), ptx::make_desc_k128(sk + k4 * 32), idesc_s, k4 ? 1u : 0u);
        ptx::tc_commit(ptx::smem_u32(&sfull_bar[w]));
      };
      auto issue_pv = [&](int j) {
        const int slot = j % kSlots, w = j & 1, i = j >> 1, r = j & 3;
        ptx::mbar_wait(ptx::smem_u32(&pready_bar[w]), i & 1);
        ptx::mbar_wait(ptx::smem_u32(&ofree_bar[r]), ((i >> 1) & 1) ^ 1);  // item j - 4 has left the O region
        ptx::tc_fence_after();
        const uint32_t sv = ptx::smem_u32(smem + (size_t)slot * kSlotBytes) + 2 * kTileBytes;
        const uint32_t d = tmem_base + (uint32_t)(kOBase + r * HD);
        const uint32_t a = tmem_base + (uint32_t)(w * kTile);
#pragma unroll
        for (int ks = 0; ks < kTile / 16; ++ks)  // 16 keys per MMA: two 8-key groups, 1024 bytes apart
          ptx::mma_ts(d, a + (uint32_t)(ks * 8), ptx::make_desc_k128(sv + ks * 2048), idesc_o, ks ? 1u : 0u);
        ptx::tc_commit(ptx::smem_u32(&ofull_bar[r]));
        ptx::tc_commit(ptx::smem_u32(&empty_bar[slot]));
      };
      if (n_local > 0) issue_s(0);
      if (n_local > 1) issue_s(1);
      for (int j = 0; j < n_local; ++j) {
        issue_pv(j);
        // S of the warpgroup's next item overwrites the P just consumed: issued behind P V on the same pipe
        if (j + 2 < n_local) issue_s(j + 2);
      }
    }
  } else {
    // ===================== softmax warpgroups =====================
    const int wg = (warp - 2) >> 2;
    const int quarter = warp & 3;
    const int r = 32 * quarter + lane;  // row of the tile == TMEM lane
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * quarter) << 16);
    const int g = p.QT > 0 ? 0 : r / p.S;
    const float sc = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e): softmax in base 2
    const uint32_t s_addr = lane_addr + (uint32_t)(wg * kTile);  // this warpgroup's S region; P = its first 64 columns
    // epilogue of an earlier item: O from TMEM, scale by 1 / row sum, bf16 into the warpgroup's staging box
    // (row = 128 bytes, 16-byte chunk c at chunk c ^ (row & 7): conflict-free), one TMA store of the box
    unsigned char* my_stage = stage_o + wg * kTileBytes;
    const uint32_t stage_u32 = ptx::smem_u32(my_stage);
    unsigned char* my_row = my_stage + r * 128;
    const int sw = r & 7;
    const bool leader = quarter == 0 && lane == 0;
    auto wg_sync = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(wg + 1) : "memory"); };
    auto epilogue = [&](int j, float inv, int row0, int head) {
      const int rgn = j & 3;
      ptx::mbar_wait(ptx::smem_u32(&ofull_bar[rgn]), (uint32_t)(j >> 2) & 1);
      ptx::tc_fence_after();
      uint32_t ov[HD];
      const uint32_t o_addr = lane_addr + (uint32_t)(kOBase + rgn * HD);
      ptx::tmem_ld_32x32b_x32(o_addr, ov);
      ptx::tmem_ld_32x32b_x32(o_addr + 32, ov + 32);
      ptx::tmem_ld_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(ptx::smem_u32(&ofree_bar[rgn]));
      if (leader) ptx::tma_store_wait_read<0>();  // the previous box of this warpgroup has left shared memory
      wg_sync();
#pragma unroll
      for (int c = 0; c < HD / 8; ++c) {
        uint4 o;
        o.x = pack_bf16(__uint_as_float(ov[c * 8 + 0]) * inv, __uint_as_float(ov[c * 8 + 1]) * inv);
        o.y = pack_bf16(__uint_as_float(ov[c * 8 + 2]) * inv, __uint_as_float(ov[c * 8 + 3]) * inv);
        o.z = pack_bf16(__uint_as_float(ov[c * 8 + 4]) * inv, __uint_as_float(ov[c * 8 + 5]) * inv);
        o.w = pack_bf16(__uint_as_float(ov[c * 8 + 6]) * inv, __uint_as_float(ov[c * 8 + 7]) * inv);
        *reinterpret_cast<uint4*>(my_row + ((c ^ sw) << 4)) = o;
      }
      ptx::fence_proxy_async_smem();
      wg_sync();
#ifdef ICD_PROFILING
      if (leader && !(p.dbg & 1)) {
#else
      if (leader) {
#endif
        // the box is G * S rows tall (the rows this tile owns); rows past the end of the buffer are clipped
        ptx::tma_store_2d(&tmap_ctx, stage_u32, head * HD, row0);
        ptx::tma_store_commit();
      }
    };
    int prev = -1, prev_row0 = 0, prev_head = 0;
    float prev_inv = 0.f;
    // the sequence length of this row for item j, requested one item ahead
    auto load_len = [&](int j) {
      const int item = (int)blockIdx.x + j * (int)gridDim.x;
      const int seq = p.QT > 0 ? (item / kHeads) / (p.QT * p.QT) : (item / kHeads) * p.G + g;
      return (j < n_local && g < p.G && seq < p.B) ? __ldg(p.lens + seq) : 0;
    };
    int next_len = load_len(wg);
    for (int j = wg; j < n_local; j += 2) {
      const int item = (int)blockIdx.x + j * (int)gridDim.x;
      const int tile = item / kHeads, head = item % kHeads;
      const uint32_t par = (uint32_t)(j >> 1) & 1;
      const int seq = p.QT > 0 ? tile / (p.QT * p.QT) : tile * p.G + g;
      const int qt = p.QT > 0 ? (tile / p.QT) % p.QT : 0, kt = p.QT > 0 ? tile % p.QT : 0;
      const bool row_used = g < p.G && seq < p.B;
      const int len = row_used ? min(next_len, p.S) : 0;
      next_len = load_len(j + 2);
      // key columns this row attends to: its own sequence inside a packed tile, or (split-KV) what the key tile holds
      const int lo = p.QT > 0 ? 0 : g * p.S;
      const int hi = p.QT > 0 ? max(0, min(kTile, len - kt * kTile)) : lo + len;
      const bool q_live = row_used && (p.QT > 0 ? (qt * kTile + r) < len : (r - lo) < len);
      // warp-uniform view of the key range: a 32-column chunk is `live` if some row of the warp needs it and
      // `full` if every row needs all of it (then no per-element mask: the common case of unpadded sequences)
      const int wlo = __reduce_min_sync(0xffffffffu, lo), whi = __reduce_max_sync(0xffffffffu, hi);
      const int wlo_max = __reduce_max_sync(0xffffffffu, lo), whi_min = __reduce_min_sync(0xffffffffu, hi);

      ptx::mbar_wait(ptx::smem_u32(&sfull_bar[wg]), par);
      ptx::tc_fence_after();
      // Two passes over the row, 64 columns (two chunks) at a time, re-reading S from TMEM for the second one: keeping
      // all 128 scores in registers cost 340 bytes of spills per thread, and TMEM reads are cheap.  Pass 2 writes P
      // chunk c (16 packed columns at 16 c) over S columns that this pass has already pulled into registers.
      auto live = [&](int c32) { return c32 * 32 < whi && c32 * 32 + 32 > wlo; };
      auto full = [&](int c32) { return c32 * 32 >= wlo_max && c32 * 32 + 32 <= whi_min; };
      auto masked = [&](uint32_t bits, int col) {
        return (col >= lo && col < hi) ? __uint_as_float(bits) : -INFINITY;
      };
      float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};  // independent chains: the reduction is latency-bound
#pragma unroll 1
      for (int h2 = 0; h2 < 2; ++h2) {
        if (!live(2 * h2) && !live(2 * h2 + 1)) continue;
        uint32_t sv[64];
        ptx::tmem_ld_32x32b_x32(s_addr + h2 * 64, sv);  // both chunks of a live pair: a dead one costs nothing to read
        ptx::tmem_ld_32x32b_x32(s_addr + h2 * 64 + 32, sv + 32);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int c32 = 2 * h2 + q;
          if (!live(c32)) continue;
          if (full(c32)) {
#pragma unroll
            for (int c = 0; c < 32; ++c) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(sv[q * 32 + c]));
          } else {
#pragma unroll
            for (int c = 0; c < 32; ++c) m4[c & 3] = fmaxf(m4[c & 3], masked(sv[q * 32 + c], c32 * 32 + c));
          }
        }
      }
      const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
      const float msc = (m == -INFINITY) ? 0.f : m * sc;
      float sum4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
      for (int h2 = 0; h2 < 2; ++h2) {
        uint32_t pk[32];
        if (live(2 * h2) || live(2 * h2 + 1)) {
          uint32_t sv[64];
          ptx::tmem_ld_32x32b_x32(s_addr + h2 * 64, sv);
          ptx::tmem_ld_32x32b_x32(s_addr + h2 * 64 + 32, sv + 32);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const int c32 = 2 * h2 + q;
            if (!live(c32)) {
#pragma unroll
              for (int c = 0; c < 16; ++c) pk[q * 16 + c] = 0u;
            } else if (full(c32)) {
#pragma unroll
              for (int c = 0; c < 16; ++c) {
                const float e0 = ex2_approx(fmaf(__uint_as_float(sv[q * 32 + 2 * c]), sc, -msc));
                const float e1 = ex2_approx(fmaf(__uint_as_float(sv[q * 32 + 2 * c + 1]), sc, -msc));
                sum4[c & 3] += e0 + e1;
                pk[q * 16 + c] = pack_bf16(e0, e1);
              }
            } else {
#pragma unroll
              for (int c = 0; c < 16; ++c) {  // masked entries are -inf: ex2 gives 0
                const float e0 = ex2_approx(fmaf(masked(sv[q * 32 + 2 * c], c32 * 32 + 2 * c), sc, -msc));
                const float e1 = ex2_approx(fmaf(masked(sv[q * 32 + 2 * c + 1], c32 * 32 + 2 * c + 1), sc, -msc));
                sum4[c & 3] += e0 + e1;
                pk[q * 16 + c] = pack_bf16(e0, e1);
              }
            }
          }
        } else {
#pragma unroll
          for (int c = 0; c < 32; ++c) pk[c] = 0u;
        }
        ptx::tmem_st_32x32b_x16(s_addr + h2 * 32, pk);
        ptx::tmem_st_32x32b_x16(s_addr + h2 * 32 + 16, pk + 16);
      }
      const float sum = (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]);
      ptx::tmem_st_wait();
      ptx::tc_fence_before();
      ptx::mbar_arrive(ptx::smem_u32(&pready_bar[wg]));

      // while P V (j) and Q K^T (j + 2) run: drain the previous item of this warpgroup
      if (prev >= 0) epilogue(prev, prev_inv, prev_row0, prev_head);
      prev = j;
      // padded query positions are never read downstream (masked keys, masked pooling): zeros
      prev_inv = (q_live && sum > 0.f) ? 1.0f / sum : 0.f;
      prev_row0 = tile * p.G * p.S;
      if (p.QT > 0) {
        // partial of (query tile, key tile): rows of key tile kt start at kt * B * S_pad in the partial buffers
        const int prow = seq * p.S_pad + qt * kTile;
        prev_row0 = kt * p.B * p.S_pad + prow;
        p.part_stats[((size_t)kt * kHeads + head) * ((size_t)p.B * p.S_pad) + prow + r] =
            make_float2(msc, (q_live && sum > 0.f) ? sum : 0.f);
      }
      prev_head = head;
    }
    if (prev >= 0) epilogue(prev, prev_inv, prev_row0, prev_head);
    if (leader) ptx::tma_store_wait_all();  // global writes complete before the kernel ends
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// merges the <= 4 key-tile partials of every (token, head): out = sum_t w_t O_t / sum_t w_t, w_t = exp2(m_t - max m) sum_t.
// One thread per (token, head, 8-column chunk) -- H / 8 threads; rows are read / written 16 bytes at a time.
template <int H>
__global__ void __launch_bounds__(H / 8)
attention_combine_kernel(const __nv_bfloat16* __restrict__ part, const float2* __restrict__ stats, int B, int S, int S_pad,
                         int QT, __nv_bfloat16* __restrict__ ctx) {
  ptx::griddep_launch();
  ptx::griddep_wait();
  constexpr int kHeads = H / HD;
  const int row = blockIdx.x;            // token row of the [B * S, H] ctx buffer
  const int seq = row / S, t = row % S;
  const int head = threadIdx.x >> 3, chunk = threadIdx.x & 7;
  const size_t prow = (size_t)seq * S_pad + t;
  const size_t plane = (size_t)B * S_pad;
  float m = -INFINITY;
  float2 st[4];
  for (int kt = 0; kt < QT; ++kt) {
    st[kt] = stats[((size_t)kt * kHeads + head) * plane + prow];
    if (st[kt].y > 0.f) m = fmaxf(m, st[kt].x);
  }
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float wsum = 0.f;
  for (int kt = 0; kt < QT; ++kt) {
    if (!(st[kt].y > 0.f)) continue;
    const float w = ex2_approx(st[kt].x - m) * st[kt].y;
    wsum += w;
    const uint4 v = *reinterpret_cast<const uint4*>(part + ((size_t)kt * plane + prow) * H + head * HD + chunk * 8);
    acc[0] = fmaf(w, bf16lo_to_f32(v.x), acc[0]); acc[1] = fmaf(w, bf16hi_to_f32(v.x), acc[1]);
    acc[2] = fmaf(w, bf16lo_to_f32(v.y), acc[2]); acc[3] = fmaf(w, bf16hi_to_f32(v.y), acc[3]);
    acc[4] = fmaf(w, bf16lo_to_f32(v.z), acc[4]); acc[5] = fmaf(w, bf16hi_to_f32(v.z), acc[5]);
    acc[6] = fmaf(w, bf16lo_to_f32(v.w), acc[6]); acc[7] = fmaf(w, bf16hi_to_f32(v.w), acc[7]);
  }
  const float inv = wsum > 0.f ? 1.0f / wsum : 0.f;
  uint4 o;
  o.x = pack_bf16(acc[0] * inv, acc[1] * inv);
  o.y = pack_bf16(acc[2] * inv, acc[3] * inv);
  o.z = pack_bf16(acc[4] * inv, acc[5] * inv);
  o.w = pack_bf16(acc[6] * inv, acc[7] * inv);
  *reinterpret_cast<uint4*>(ctx + (size_t)row * H + head * HD + chunk * 8) = o;
}

}  // namespace

static bool supported_hidden(int hidden) {
  if (hidden == 768 || hidden == 1024) return true;
  set_error("attention: hidden size %d is not supported (768 or 1024)", hidden);
  return false;
}

int attention_make_map(void* map128, const void* qkv, int64_t rows, int hidden) {
  if (!supported_hidden(hidden)) return ICD_E_ARG;
  return make_tmap_bf16_2d(map128, qkv, (uint64_t)rows, (uint64_t)(3 * hidden), kTile, HD, true);
}

template <int H>
static int launch_packed(const CUtensorMap& tm, const AttParams& p, void* ctx, int64_t ctx_rows, cudaStream_t st) {
  // ctx store box: the G * S rows a tile owns x one head (64 columns); encoded per launch because it depends on S
  alignas(128) unsigned char ctx_map[128];
  ICD_TRY(make_tmap_bf16_2d(ctx_map, ctx, (uint64_t)ctx_rows, (uint64_t)H, (uint32_t)(p.G * p.S), HD, true));
  CUtensorMap tc;
  memcpy(&tc, ctx_map, sizeof(tc));
  ICD_CUDA(cudaFuncSetAttribute(attention_tc_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int grid = std::min(p.tiles * (H / HD), kSMs);
  ICD_CUDA(launch_chained(attention_tc_kernel<H>, dim3(grid), dim3(kThreads), (size_t)kSmemBytes, st, 1, tm, tc, p));
  count_launch();
  return ICD_OK;
}

int launch_attention_tc(const void* tmap_qkv, const int32_t* lens, int B, int S, void* ctx, int64_t ctx_rows,
                        cudaStream_t st, int hidden) {
  if (S < 1 || S > kTile) {
    set_error("attention: S=%d outside [1, 128]", S);
    return ICD_E_UNSUPPORTED;
  }
  if (!supported_hidden(hidden)) return ICD_E_ARG;
  AttParams p{};
  p.lens = lens;
  p.B = B;
  p.S = S;
  p.G = kTile / S;
  p.tiles = (B + p.G - 1) / p.G;
#ifdef ICD_PROFILING
  {
    static const int dbg = getenv("ICD_ATTN_DBG") ? atoi(getenv("ICD_ATTN_DBG")) : 0;
    p.dbg = dbg;
  }
#endif
  CUtensorMap tm;
  memcpy(&tm, tmap_qkv, sizeof(tm));
  return hidden == 768 ? launch_packed<768>(tm, p, ctx, ctx_rows, st) : launch_packed<1024>(tm, p, ctx, ctx_rows, st);
}

// split-KV form for 128 < S <= 512: part [QT * B * S_pad, H] bf16 and stats [QT * heads * B * S_pad] float2 are scratch
size_t attention_long_scratch_bytes(int B, int S, size_t* stats_bytes, int hidden) {
  const int QT = (S + kTile - 1) / kTile;
  const size_t rows = (size_t)QT * B * QT * kTile;
  if (stats_bytes) *stats_bytes = (size_t)QT * (hidden / HD) * B * QT * kTile * sizeof(float2);
  return rows * hidden * 2;
}

template <int H>
static int launch_split(const CUtensorMap& tm, const AttParams& p, void* part, void* ctx, cudaStream_t st) {
  alignas(128) unsigned char part_map[128];
  ICD_TRY(make_tmap_bf16_2d(part_map, part, (uint64_t)p.QT * p.B * p.S_pad, (uint64_t)H, (uint32_t)kTile, HD, true));
  CUtensorMap tc;
  memcpy(&tc, part_map, sizeof(tc));
  ICD_CUDA(cudaFuncSetAttribute(attention_tc_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
  const int grid = std::min(p.tiles * (H / HD), kSMs);
  ICD_CUDA(launch_chained(attention_tc_kernel<H>, dim3(grid), dim3(kThreads), (size_t)kSmemBytes, st, 1, tm, tc, p));
  count_launch();
  ICD_CUDA(launch_chained(attention_combine_kernel<H>, dim3(p.B * p.S), dim3(H / 8), 0, st, 1,
                          reinterpret_cast<const __nv_bfloat16*>(part), static_cast<const float2*>(p.part_stats), p.B, p.S,
                          p.S_pad, p.QT, reinterpret_cast<__nv_bfloat16*>(ctx)));
  count_launch();
  return ICD_OK;
}

int launch_attention_tc_long(const void* tmap_qkv, const int32_t* lens, int B, int S, void* part, void* stats, void* ctx,
                             cudaStream_t st, int hidden) {
  if (S <= kTile || S > 4 * kTile) {
    set_error("attention (split-KV): S=%d outside (128, 512]", S);
    return ICD_E_UNSUPPORTED;
  }
  if (!supported_hidden(hidden)) return ICD_E_ARG;
  AttParams p{};
  p.lens = lens;
  p.B = B;
  p.S = S;
  p.G = 1;
  p.QT = (S + kTile - 1) / kTile;
  p.S_pad = p.QT * kTile;
  p.tiles = B * p.QT * p.QT;
  p.part_stats = reinterpret_cast<float2*>(stats);
  CUtensorMap tm;
  memcpy(&tm, tmap_qkv, sizeof(tm));
  return hidden == 768 ? launch_split<768>(tm, p, part, ctx, st) : launch_split<1024>(tm, p, part, ctx, st);
}

}  // namespace icd
