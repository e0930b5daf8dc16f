// topk_large.cu -- exact paged search beyond ICD_MAX_K (icd_index_search_page): offset + limit up to ICD_MAX_LIMIT,
// Milvus range search on the raw inner product.
//
// The scan paths keep candidate lists of at most ICD_MAX_K rows, so a long list takes a different road, exact by
// construction, and every buffer it writes is sized on the host before the launch:
//   page_score_kernel   canonical fp32 score (canon_dot.cuh) of every (query, row) of a query chunk -> [Bc, n] raw
//                       workspace; a row the mask or the range excludes gets a sentinel below every real key
//   page_hist_kernel /  radix select of the K-th largest order-preserving key per query, 8 bits per pass over four
//   page_choose_kernel  passes; histograms from (row block, query) CTAs
//   page_count_kernel / per-block counts of the rows above the K-th key and of the rows equal to it, an exclusive scan
//   page_scan_kernel /  over the blocks, then each block writes its rows at its offsets: the ties taken are the
//   page_gather_kernel  lowest ids, and no write lands at or past K (every position is checked against the host's K)
//   page_final_kernel   per query: bitonic sort of the <= K (key, id) pairs in shared memory, the weight rule, the page
#include <algorithm>

#include "canon_dot.cuh"
#include "common.cuh"
#include "kernels.h"

namespace icd {
namespace {

constexpr uint32_t kSentinelBits = 0xffffffffu;  // a NaN no FMA produces: "this row may not be returned"
constexpr int kScoreQ = 8;                       // queries per score CTA (one row read serves all of them); 1 for B = 1
constexpr int kScoreWarps = 8;
constexpr int kSelThreads = 256;
constexpr int kSelRows = 8192;                   // contiguous rows per select CTA
constexpr int kFinalThreads = 1024;
constexpr size_t kWorkspaceBudget = 512ull << 20;   // bytes of [Bc, n] raw scores (and the rest) per query chunk

// Order-preserving selection key of a raw score: key(a) > key(b) <=> a > b, with -0.0 and +0.0 one key (cand_before
// calls them equal and breaks the tie by id).  Real keys are >= 1; 0 is the sentinel.  WEIGHT_PRE selects on the fp32
// raw * w(level), as finalise_kernel does.
__device__ __forceinline__ uint32_t sel_key(uint32_t bits, uint8_t lv, bool pre) {
  if (bits == kSentinelBits) return 0u;
  float k = __uint_as_float(bits);
  if (pre) k = k * level_weight_f(lv);
  if (k == 0.f) k = 0.f;
  uint32_t u = __float_as_uint(k);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return max(u, 1u);
}

// exclusive scan of one uint64 per thread over the block (blockDim.x a multiple of 32); *total = the block's sum
__device__ __forceinline__ uint64_t block_excl_scan(uint64_t v, uint64_t* total) {
  __shared__ uint64_t s_w[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  uint64_t inc = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const uint64_t o = __shfl_up_sync(0xffffffffu, inc, off);
    if (lane >= off) inc += o;
  }
  if (lane == 31) s_w[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = lane < nw ? s_w[lane] : 0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const uint64_t o = __shfl_up_sync(0xffffffffu, w, off);
      if (lane >= off) w += o;
    }
    if (lane < nw) s_w[lane] = w;   // inclusive totals of the warps
  }
  __syncthreads();
  const uint64_t base = warp ? s_w[warp - 1] : 0;
  *total = s_w[nw - 1];
  __syncthreads();   // s_w is reused by the next call
  return base + inc - v;
}

// Scores of NQ queries against every row.  A warp takes 32 consecutive rows and keeps row r's scores in lane r, so
// each query's 32 scores leave as one coalesced store.
template <bool F32ROWS, int CPL, int NQ>
__global__ void __launch_bounds__(kScoreWarps * 32, 2)
page_score_kernel(const void* __restrict__ rows, int64_t n, int dim, const float* __restrict__ q, int nq,
                  const uint32_t* __restrict__ mask, int range_flags, float radius, float range_filter,
                  float* __restrict__ ws) {
  extern __shared__ __align__(16) float s_q[];   // [NQ][dim]
  constexpr int E = F32ROWS ? 4 : 8;
  const int q0 = blockIdx.y * NQ;
  const int nqv = min(NQ, nq - q0);
  for (int i = threadIdx.x; i < NQ * dim; i += blockDim.x) {
    const int j = i / dim;
    s_q[i] = j < nqv ? q[(size_t)(q0 + j) * dim + (i - j * dim)] : 0.f;
  }
  __syncthreads();
  const int nchunks = dim / E;
  const size_t row_bytes = (size_t)dim * (F32ROWS ? 4 : 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const char* base = reinterpret_cast<const char*>(rows);
  for (int64_t r0 = ((int64_t)blockIdx.x * kScoreWarps + warp) * 32; r0 < n;
       r0 += (int64_t)gridDim.x * kScoreWarps * 32) {
    const uint32_t mbits = mask ? __ldg(mask + (r0 >> 5)) : 0xffffffffu;   // r0 is a multiple of 32
    const int rn = n - r0 < 32 ? (int)(n - r0) : 32;
    float mine[NQ];
#pragma unroll
    for (int j = 0; j < NQ; ++j) mine[j] = 0.f;
    for (int r = 0; r < rn; ++r) {
      if (!((mbits >> r) & 1u)) continue;   // warp-uniform
      const char* rp = base + (size_t)(r0 + r) * row_bytes;
      uint4 v[CPL];
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = lane + 32 * i;
        v[i] = c < nchunks ? *reinterpret_cast<const uint4*>(rp + (size_t)c * 16) : make_uint4(0, 0, 0, 0);
      }
      float acc[NQ];
#pragma unroll
      for (int j = 0; j < NQ; ++j) acc[j] = 0.f;
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = lane + 32 * i;
        if (c < nchunks) {
#pragma unroll
          for (int j = 0; j < NQ; ++j) acc[j] = canon_chunk_fma<F32ROWS>(v[i], s_q + j * dim + c * E, acc[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < NQ; ++j) {
        const float s = canon_lane_sum(acc[j]);
        if (lane == r) mine[j] = s;
      }
    }
    if (lane < rn) {
      const bool allowed = (mbits >> lane) & 1u;
#pragma unroll
      for (int j = 0; j < NQ; ++j) {
        if (j >= nqv) break;
        const float s = mine[j];
        bool keep = allowed;
        if (range_flags & ICD_RANGE_RADIUS) keep = keep && s > radius;
        if (range_flags & ICD_RANGE_FILTER) keep = keep && s <= range_filter;
        ws[(size_t)(q0 + j) * n + r0 + lane] = keep ? s : __uint_as_float(kSentinelBits);
      }
    }
  }
}

// histogram of digit `pass` (8 bits, most significant first) over the keys that match the prefix chosen so far
__global__ void __launch_bounds__(kSelThreads)
page_hist_kernel(const float* __restrict__ ws, const uint8_t* __restrict__ levels, int64_t n, int pre, int pass,
                 const uint32_t* __restrict__ state, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  const int b = blockIdx.y;
  const int shift = 24 - 8 * pass;
  const uint32_t prefix = pass ? state[(size_t)b * 4] : 0u;
  const uint32_t hi_mask = pass ? (0xffffffffu << (shift + 8)) : 0u;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(ws) + (size_t)b * n;
  const int64_t r0 = (int64_t)blockIdx.x * kSelRows, r1 = min(n, r0 + kSelRows);
  for (int64_t base = r0; base < r1; base += kSelThreads) {   // every thread takes the same trips: full-warp match
    const int64_t r = base + threadIdx.x;
    uint32_t bin = 256;
    if (r < r1) {
      const uint32_t key = sel_key(w[r], pre ? levels[r] : (uint8_t)0, pre != 0);
      if ((key & hi_mask) == prefix) bin = (key >> shift) & 255u;
    }
    const uint32_t peers = __match_any_sync(0xffffffffu, bin);
    if (bin < 256 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[bin], (uint32_t)__popc(peers));
  }
  __syncthreads();
  const uint32_t c = h[threadIdx.x];
  if (c) atomicAdd(&hist[(size_t)b * 256 + threadIdx.x], c);
}

// per query: the bin holding the krem-th largest key of the prefix group; clears the histogram for the next pass.
// state[b] = {prefix (the K-th key after the last pass), krem, rows above the K-th key taken, rows taken}
__global__ void __launch_bounds__(256)
page_choose_kernel(uint32_t* __restrict__ hist, uint32_t* __restrict__ state, int pass, uint32_t K) {
  __shared__ uint32_t h[256];
  const int b = blockIdx.x;
  h[threadIdx.x] = hist[(size_t)b * 256 + threadIdx.x];
  hist[(size_t)b * 256 + threadIdx.x] = 0;
  __syncthreads();
  if (threadIdx.x == 0) {
    const uint32_t krem = pass ? state[(size_t)b * 4 + 1] : K;
    const uint32_t prefix = pass ? state[(size_t)b * 4] : 0u;
    uint32_t cum = 0;
    int bin = 255;
    for (; bin > 0; --bin) {
      if (cum + h[bin] >= krem) break;
      cum += h[bin];
    }
    state[(size_t)b * 4] = prefix | ((uint32_t)bin << (24 - 8 * pass));
    state[(size_t)b * 4 + 1] = krem - cum;
  }
}

__global__ void __launch_bounds__(kSelThreads)
page_count_kernel(const float* __restrict__ ws, const uint8_t* __restrict__ levels, int64_t n, int pre,
                  const uint32_t* __restrict__ state, uint2* __restrict__ cnt, int nblk) {
  __shared__ uint32_t s_g[kSelThreads / 32], s_e[kSelThreads / 32];
  const int b = blockIdx.y;
  const uint32_t kth = state[(size_t)b * 4];
  const uint32_t* w = reinterpret_cast<const uint32_t*>(ws) + (size_t)b * n;
  const int64_t r0 = (int64_t)blockIdx.x * kSelRows, r1 = min(n, r0 + kSelRows);
  uint32_t g = 0, e = 0;
  for (int64_t r = r0 + threadIdx.x; r < r1; r += kSelThreads) {
    const uint32_t key = sel_key(w[r], pre ? levels[r] : (uint8_t)0, pre != 0);
    g += key > kth ? 1u : 0u;
    e += key == kth ? 1u : 0u;
  }
  g = __reduce_add_sync(0xffffffffu, g);
  e = __reduce_add_sync(0xffffffffu, e);
  if ((threadIdx.x & 31) == 0) s_g[threadIdx.x >> 5] = g, s_e[threadIdx.x >> 5] = e;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tg = 0, te = 0;
    for (int i = 0; i < kSelThreads / 32; ++i) tg += s_g[i], te += s_e[i];
    cnt[(size_t)b * nblk + blockIdx.x] = make_uint2(tg, te);
  }
}

// per query: exclusive offsets of every block's rows above / at the K-th key, and how many of each the list takes
__global__ void __launch_bounds__(kFinalThreads)
page_scan_kernel(const uint2* __restrict__ cnt, uint2* __restrict__ off, int nblk, uint32_t* __restrict__ state,
                 uint32_t K) {
  const int b = blockIdx.x;
  uint64_t run = 0;   // (eq << 32) | gt of the blocks before this tile
  for (int base = 0; base < nblk; base += kFinalThreads) {
    const int i = base + threadIdx.x;
    const uint2 c = i < nblk ? cnt[(size_t)b * nblk + i] : make_uint2(0, 0);
    uint64_t total;
    const uint64_t ex = block_excl_scan(((uint64_t)c.y << 32) | c.x, &total) + run;
    if (i < nblk) off[(size_t)b * nblk + i] = make_uint2((uint32_t)ex, (uint32_t)(ex >> 32));
    run += total;
  }
  if (threadIdx.x == 0) {
    const uint32_t kth = state[(size_t)b * 4];
    const uint32_t gt = min((uint32_t)run, K), eq = (uint32_t)(run >> 32);
    const uint32_t ties = kth > 0 ? min(eq, K - gt) : 0u;   // key 0: the sentinel rows, never returned
    state[(size_t)b * 4 + 2] = gt;
    state[(size_t)b * 4 + 3] = gt + ties;
  }
}

__global__ void __launch_bounds__(kSelThreads)
page_gather_kernel(const float* __restrict__ ws, const uint8_t* __restrict__ levels, int64_t n, int pre,
                   const uint32_t* __restrict__ state, const uint2* __restrict__ off, int nblk, int K,
                   int* __restrict__ cand) {
  __shared__ uint32_t s_g[kSelThreads / 32], s_e[kSelThreads / 32];
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t kth = state[(size_t)b * 4], gt_total = state[(size_t)b * 4 + 2];
  const uint32_t ties = state[(size_t)b * 4 + 3] - gt_total;
  const uint2 o = off[(size_t)b * nblk + blockIdx.x];
  uint32_t gbase = o.x, ebase = o.y;
  const uint32_t* w = reinterpret_cast<const uint32_t*>(ws) + (size_t)b * n;
  int* out = cand + (size_t)b * K;
  const uint32_t lt = (1u << lane) - 1u;
  const int64_t r0 = (int64_t)blockIdx.x * kSelRows, r1 = min(n, r0 + kSelRows);
  for (int64_t base = r0; base < r1; base += kSelThreads) {
    const int64_t r = base + threadIdx.x;
    uint32_t key = 0;
    if (r < r1) key = sel_key(w[r], pre ? levels[r] : (uint8_t)0, pre != 0);
    const bool g = r < r1 && key > kth;
    const bool e = r < r1 && kth > 0 && key == kth;
    const uint32_t bg = __ballot_sync(0xffffffffu, g), be = __ballot_sync(0xffffffffu, e);
    if (lane == 0) s_g[warp] = __popc(bg), s_e[warp] = __popc(be);
    __syncthreads();
    uint32_t pg = 0, pe = 0, tg = 0, te = 0;
#pragma unroll
    for (int i = 0; i < kSelThreads / 32; ++i) {
      if (i < warp) pg += s_g[i], pe += s_e[i];
      tg += s_g[i], te += s_e[i];
    }
    if (g) {
      const uint32_t pos = gbase + pg + __popc(bg & lt);
      if (pos < gt_total) out[pos] = (int)r;
    }
    if (e) {
      const uint32_t t = ebase + pe + __popc(be & lt);
      if (t < ties) out[gt_total + t] = (int)r;
    }
    gbase += tg;
    ebase += te;
    __syncthreads();
  }
}

struct FinalArgs {
  const int* cand;   // [Bc, K]
  const float* ws;   // [Bc, n]
  const uint8_t* levels;
  int64_t n;
  const uint32_t* state;
  int K, Kp, weight_mode, offset, limit;
  float* out_score;  // [Bc, limit] each, may be null
  float* out_raw;
  int64_t* out_id;
};

__device__ __forceinline__ int weight_class(uint8_t lv) { return lv == 1 ? 0 : (lv == 3 ? 2 : 1); }
__device__ __forceinline__ double class_weight(int c) { return c == 0 ? 1.2 : (c == 2 ? 0.8 : 1.0); }

// one CTA per query: sort the list, apply the weight rule, write the page [offset, offset + limit)
__global__ void __launch_bounds__(kFinalThreads)
page_final_kernel(FinalArgs a) {
  extern __shared__ __align__(16) unsigned long long s_list[];   // [Kp]: (key << 32) | ~id, later (raw bits << 32) | id
  uint16_t* runs = reinterpret_cast<uint16_t*>(s_list + a.Kp);  // [K]: list positions grouped by level class
  const int b = blockIdx.x;
  const uint32_t kout = a.state[(size_t)b * 4 + 3];
  const bool pre = a.weight_mode == ICD_WEIGHT_PRE;
  const float* w = a.ws + (size_t)b * a.n;
  const int* cand = a.cand + (size_t)b * a.K;
  for (int p = threadIdx.x; p < a.Kp; p += blockDim.x) {
    unsigned long long v = 0;
    if (p < (int)kout) {
      const uint32_t id = min((uint32_t)cand[p], (uint32_t)(a.n - 1));   // every slot below kout was gathered
      const uint32_t key = sel_key(__float_as_uint(w[id]), a.levels[id], pre);
      v = ((unsigned long long)key << 32) | (uint32_t)~id;
    }
    s_list[p] = v;
  }
  __syncthreads();
  // bitonic sort, descending: (key desc, id asc); the zero padding sinks to the end
  for (int k2 = 2; k2 <= a.Kp; k2 <<= 1) {
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < a.Kp; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = s_list[i], y = s_list[ixj];
          if (((i & k2) == 0) ? (x < y) : (x > y)) {
            s_list[i] = y;
            s_list[ixj] = x;
          }
        }
      }
      __syncthreads();
    }
  }
  const size_t orow = (size_t)b * a.limit;
  auto put = [&](int slot, float score, float raw, int64_t id) {
    if (a.out_score) a.out_score[orow + slot] = score;
    if (a.out_raw) a.out_raw[orow + slot] = raw;
    if (a.out_id) a.out_id[orow + slot] = id;
  };
  for (int j = threadIdx.x; j < a.limit; j += blockDim.x)
    if ((int64_t)a.offset + j >= (int64_t)kout) put(j, -INFINITY, -INFINITY, -1);

  if (a.weight_mode != ICD_WEIGHT_RERANK) {
    for (int j = threadIdx.x; j < a.limit; j += blockDim.x) {
      const int p = a.offset + j;
      if (p >= (int)kout) continue;
      const uint32_t id = ~(uint32_t)s_list[p];
      const float raw = w[id];
      put(j, pre ? raw * level_weight_f(a.levels[id]) : raw, raw, (int64_t)id);
    }
    return;
  }

  // WEIGHT_RERANK: the reference's stable re-sort of the whole list by double(raw) * w(level).  The list is in raw order,
  // so the positions of each level class form a run already in re-sorted order; an element's rank is its index in its
  // own run plus, for each other run, how many of that run's elements precede it (a prefix: binary search).
  const int seg = (a.Kp + blockDim.x - 1) / blockDim.x;
  const int p0 = threadIdx.x * seg, p1 = min((int)kout, p0 + seg);
  uint64_t mine = 0;
  for (int p = p0; p < p1; ++p) {
    const uint32_t id = ~(uint32_t)s_list[p];
    const uint32_t bits = __float_as_uint(w[id]);
    mine += 1ull << (21 * weight_class(a.levels[id]));
    s_list[p] = ((unsigned long long)bits << 32) | id;
  }
  uint64_t total;
  uint64_t at = block_excl_scan(mine, &total);
  const int cnt0 = (int)(total & 0x1fffff), cnt1 = (int)((total >> 21) & 0x1fffff), cnt2 = (int)(total >> 42);
  const int start[3] = {0, cnt0, cnt0 + cnt1};
  const int count[3] = {cnt0, cnt1, cnt2};
  for (int p = p0; p < p1; ++p) {
    const int c = weight_class(a.levels[(uint32_t)s_list[p]]);
    const int idx = (int)((at >> (21 * c)) & 0x1fffff);
    runs[start[c] + idx] = (uint16_t)p;
    at += 1ull << (21 * c);
  }
  __syncthreads();
  for (int c = 0; c < 3; ++c) {
    for (int i = threadIdx.x; i < count[c]; i += blockDim.x) {
      const int p = runs[start[c] + i];
      const unsigned long long e = s_list[p];
      const float raw = __uint_as_float((uint32_t)(e >> 32));
      const double tw = (double)raw * class_weight(c);
      int rank = i;
      for (int c2 = 0; c2 < 3; ++c2) {
        if (c2 == c) continue;
        const double w2 = class_weight(c2);
        int lo = 0, hi = count[c2];   // first element of run c2 that does not precede (tw, p)
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          const int p2 = runs[start[c2] + mid];
          const double t2 = (double)__uint_as_float((uint32_t)(s_list[p2] >> 32)) * w2;
          if (t2 > tw || (t2 == tw && p2 < p)) lo = mid + 1;
          else hi = mid;
        }
        rank += lo;
      }
      const int slot = rank - a.offset;
      if (slot >= 0 && slot < a.limit) put(slot, (float)tw, raw, (int64_t)(uint32_t)e);
    }
  }
}

template <bool F32ROWS, int CPL, int NQ>
int launch_score_nq(const PageSearchArgs& a, const float* q, int nq, float* ws, cudaStream_t st) {
  const int gy = (nq + NQ - 1) / NQ;
  const int64_t tiles = (a.n + 31) / 32;
  const int64_t want = (tiles + kScoreWarps - 1) / kScoreWarps;
  const int gx = (int)std::max<int64_t>(1, std::min<int64_t>(want, std::max<int64_t>(1, (int64_t)kSMs * 16 / gy)));
  const size_t smem = (size_t)NQ * a.dim * 4;
  page_score_kernel<F32ROWS, CPL, NQ><<<dim3(gx, gy), kScoreWarps * 32, smem, st>>>(
      a.rows, a.n, a.dim, q, nq, a.mask, a.range_flags, a.radius, a.range_filter, ws);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

template <bool F32ROWS, int CPL>
int launch_score(const PageSearchArgs& a, const float* q, int nq, float* ws, cudaStream_t st) {
  return nq == 1 ? launch_score_nq<F32ROWS, CPL, 1>(a, q, nq, ws, st) : launch_score_nq<F32ROWS, CPL, kScoreQ>(a, q, nq, ws, st);
}

int launch_score_any(const PageSearchArgs& a, const float* q, int nq, float* ws, cudaStream_t st) {
  if (a.f32rows) {
    switch ((a.dim / 4 + 31) / 32) {
      case 1: return launch_score<true, 1>(a, q, nq, ws, st);
      case 2: return launch_score<true, 2>(a, q, nq, ws, st);
      case 3: return launch_score<true, 3>(a, q, nq, ws, st);
      case 4: return launch_score<true, 4>(a, q, nq, ws, st);
      case 5: return launch_score<true, 5>(a, q, nq, ws, st);
      case 6: return launch_score<true, 6>(a, q, nq, ws, st);
      case 7: return launch_score<true, 7>(a, q, nq, ws, st);
      case 8: return launch_score<true, 8>(a, q, nq, ws, st);
      default: break;
    }
  } else {
    switch ((a.dim / 8 + 31) / 32) {
      case 1: return launch_score<false, 1>(a, q, nq, ws, st);
      case 2: return launch_score<false, 2>(a, q, nq, ws, st);
      case 3: return launch_score<false, 3>(a, q, nq, ws, st);
      case 4: return launch_score<false, 4>(a, q, nq, ws, st);
      default: break;
    }
  }
  set_error("page search: dim %d not supported", a.dim);
  return ICD_E_UNSUPPORTED;
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

struct Layout {
  int nblk;
  size_t ws, hist, state, cnt, off, cand, total;
};
Layout layout(int64_t n, int K, int bc) {
  Layout l{};
  l.nblk = (int)((n + kSelRows - 1) / kSelRows);
  size_t at = 0;
  l.ws = at;
  at += align256((size_t)bc * n * 4);
  l.hist = at;
  at += align256((size_t)bc * 256 * 4);
  l.state = at;
  at += align256((size_t)bc * 16);
  l.cnt = at;
  at += align256((size_t)bc * l.nblk * 8);
  l.off = at;
  at += align256((size_t)bc * l.nblk * 8);
  l.cand = at;
  at += align256((size_t)bc * K * 4);
  l.total = at;
  return l;
}

int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

}  // namespace

int page_search_chunk(int64_t n, int K, int B) {
  const size_t per_query = (size_t)n * 4 + 256 * 4 + 16 + (size_t)((n + kSelRows - 1) / kSelRows) * 16 + (size_t)K * 4;
  const size_t bc = std::max<size_t>(1, kWorkspaceBudget / per_query);
  return (int)std::min<size_t>(std::min<size_t>(bc, 65535), (size_t)std::max(B, 1));
}

size_t page_search_workspace_bytes(int64_t n, int K, int bc) { return layout(n, K, bc).total; }

int launch_page_search(const PageSearchArgs& a, cudaStream_t st) {
  const int K = a.offset + a.limit;
  if (a.limit < 1 || a.offset < 0 || K > ICD_MAX_LIMIT || a.chunk < 1 || a.n < 0 || a.n > 0x7fffffffLL) {
    set_error("page search: offset %d limit %d chunk %d n %lld", a.offset, a.limit, a.chunk, (long long)a.n);
    return ICD_E_ARG;
  }
  const Layout L = layout(a.n, K, a.chunk);
  if (L.total > a.workspace_bytes) {
    set_error("page search: workspace of %zu bytes, %zu needed", a.workspace_bytes, L.total);
    return ICD_E_ARG;
  }
  char* wsb = reinterpret_cast<char*>(a.workspace);
  float* ws = reinterpret_cast<float*>(wsb + L.ws);
  uint32_t* hist = reinterpret_cast<uint32_t*>(wsb + L.hist);
  uint32_t* state = reinterpret_cast<uint32_t*>(wsb + L.state);
  uint2* cnt = reinterpret_cast<uint2*>(wsb + L.cnt);
  uint2* off = reinterpret_cast<uint2*>(wsb + L.off);
  int* cand = reinterpret_cast<int*>(wsb + L.cand);
  const int pre = a.weight_mode == ICD_WEIGHT_PRE ? 1 : 0;
  const int Kp = next_pow2(K);
  const size_t fsmem = (size_t)Kp * 8 + (size_t)K * 2;
  ICD_CUDA(cudaFuncSetAttribute(page_final_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
  for (int q0 = 0; q0 < a.nq; q0 += a.chunk) {
    const int bc = std::min(a.chunk, a.nq - q0);
    if (a.n > 0) {
      ICD_TRY(launch_score_any(a, a.q + (size_t)q0 * a.dim, bc, ws, st));
      if (a.n > K) {
        ICD_CUDA(cudaMemsetAsync(hist, 0, (size_t)bc * 256 * 4, st));
        for (int pass = 0; pass < 4; ++pass) {
          page_hist_kernel<<<dim3(L.nblk, bc), kSelThreads, 0, st>>>(ws, a.levels, a.n, pre, pass, state, hist);
          page_choose_kernel<<<bc, 256, 0, st>>>(hist, state, pass, (uint32_t)K);
          count_launch(2);
          ICD_CUDA(cudaGetLastError());
        }
      } else {
        ICD_CUDA(cudaMemsetAsync(state, 0, (size_t)bc * 16, st));   // K-th key 0: every allowed row
      }
      page_count_kernel<<<dim3(L.nblk, bc), kSelThreads, 0, st>>>(ws, a.levels, a.n, pre, state, cnt, L.nblk);
      page_scan_kernel<<<bc, kFinalThreads, 0, st>>>(cnt, off, L.nblk, state, (uint32_t)K);
      page_gather_kernel<<<dim3(L.nblk, bc), kSelThreads, 0, st>>>(ws, a.levels, a.n, pre, state, off, L.nblk, K, cand);
      count_launch(3);
      ICD_CUDA(cudaGetLastError());
    } else {
      ICD_CUDA(cudaMemsetAsync(state, 0, (size_t)bc * 16, st));   // an empty table: an all-tail page
    }
    FinalArgs f{};
    f.cand = cand;
    f.ws = ws;
    f.levels = a.levels;
    f.n = a.n;
    f.state = state;
    f.K = K;
    f.Kp = Kp;
    f.weight_mode = a.weight_mode;
    f.offset = a.offset;
    f.limit = a.limit;
    const size_t o = (size_t)q0 * a.limit;
    f.out_score = a.out_score ? a.out_score + o : nullptr;
    f.out_raw = a.out_raw ? a.out_raw + o : nullptr;
    f.out_id = a.out_id ? a.out_id + o : nullptr;
    page_final_kernel<<<bc, kFinalThreads, fsmem, st>>>(f);
    count_launch();
    ICD_CUDA(cudaGetLastError());
  }
  return ICD_OK;
}

}  // namespace icd
