// topk_merge.cu -- reduction of per-CTA top-k lists, exact rescoring, level re-rank.
//
//   merge_kernel     [B, P, k] sorted partial lists -> [B, k]           (warp per query)
//   finalise_kernel  candidates -> exact fp32 rescoring -> sort -> cut to k -> the reference's
//                    level weighting and re-sort (services/milvus_service.py:290-314,550-558)
// Both are latency-sized (k <= 128 candidates per list); the roofline kernel is the scan.
#include "canon_dot.cuh"
#include "common.cuh"
#include "kernels.h"

namespace icd {
namespace {

constexpr int kMergeWarps = 4;
constexpr int kMaxP = 1024;

__global__ void __launch_bounds__(kMergeWarps * 32)
merge_kernel(const float* __restrict__ part_score, const int* __restrict__ part_id, int B, int P,
             int k_in, int k_out, float* __restrict__ out_score, int64_t* __restrict__ out_id,
             int64_t row_offset, int* __restrict__ bound_key_out, const int* __restrict__ count) {
  __shared__ unsigned char heads[kMergeWarps][kMaxP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kMergeWarps + warp;
  if (b >= B || (count && b >= *count)) return;
  unsigned char* hd = heads[warp];
  for (int l = lane; l < P; l += 32) hd[l] = 0;
  __syncwarp();
  const float* ps = part_score + (size_t)b * P * k_in;
  const int* pi = part_id + (size_t)b * P * k_in;

  // each lane caches the best head among the lists it owns (l = lane, lane+32, ...)
  float bs;
  int bi, bl;
  auto rescan = [&]() {
    bs = -INFINITY;
    bi = 0x7fffffff;
    bl = -1;
    for (int l = lane; l < P; l += 32) {
      const int h = hd[l];
      if (h >= k_in) continue;
      const float s = ps[(size_t)l * k_in + h];
      int id = pi[(size_t)l * k_in + h];
      if (id < 0) continue;  // empty tail of this list
      if (bl < 0 || cand_before(s, id, bs, bi)) {
        bs = s;
        bi = id;
        bl = l;
      }
    }
  };
  rescan();
  for (int j = 0; j < k_out; ++j) {
    float ws = bs;
    int wi = bi, wl = bl;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float os = __shfl_xor_sync(0xffffffffu, ws, off);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, off);
      const int ol = __shfl_xor_sync(0xffffffffu, wl, off);
      const bool take = (ol >= 0) && (wl < 0 || cand_before(os, oi, ws, wi));
      if (take) {
        ws = os;
        wi = oi;
        wl = ol;
      }
    }
    if (lane == 0) {
      out_score[(size_t)b * k_out + j] = (wl < 0) ? -INFINITY : ws;
      out_id[(size_t)b * k_out + j] = (wl < 0) ? -1 : (int64_t)wi + row_offset;
      if (bound_key_out && j == k_out - 1) bound_key_out[b] = (wl < 0) ? (int)0x80808080 : float_key(ws);
    }
    if (wl >= 0 && (wl & 31) == lane) {
      hd[wl] = hd[wl] + 1;
      rescan();
    }
  }
}

// Pre-pass bound (scan_tc.cu, PRE).  The pre-pass left one running maximum per (query, row group g, slot j) -- slot =
// accumulator column mod 32 -- and these P x 32 maxima belong to DISJOINT sets of sampled rows.  Row groups fold into
// kFolds classes (g mod kFolds), which leaves kFolds x 32 = 128 disjoint sets per query; the kc-th largest of their maxima
// is reached by >= kc distinct rows: a proven lower bound of the kc-th best score of the table, for every kc <= 128.
// (Round 2 folded all groups into one class: 32 sets, kc <= 32, and a bound at about the 1.4 kc-th best sampled score; with
// 128 sets it sits at about the 1.1 kc-th.)
constexpr int kFolds = 4;
// One block of kFolds warps per query: warp f folds the row groups of class f (lane = slot; 8 independent loads in
// flight, the chain of P dependent L2 round trips was ~30 us at small batches), the 128 maxima meet in shared memory and
// every thread ranks its own value by counting (descending, ties by index).
__global__ void __launch_bounds__(kFolds * 32)
bound_from_slots_kernel(const float* __restrict__ slot_max, int B, int P, int kc, int* __restrict__ bound_key_out) {
  __shared__ float vals[kFolds * 32];
  const int f = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x;
  const float* base = slot_max + (size_t)b * P * 32 + lane;
  float m = -INFINITY;
  int g = f;
  for (; g + 7 * kFolds < P; g += 8 * kFolds) {
    float v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = base[(size_t)(g + u * kFolds) * 32];
#pragma unroll
    for (int u = 0; u < 8; ++u) m = fmaxf(m, v[u]);
  }
  for (; g < P; g += kFolds) m = fmaxf(m, base[(size_t)g * 32]);
  vals[threadIdx.x] = m;
  __syncthreads();
  int rank = 0;
#pragma unroll 8
  for (int o = 0; o < kFolds * 32; ++o) {
    const float v = vals[o];
    rank += (v > m || (v == m && o < (int)threadIdx.x)) ? 1 : 0;
  }
  if (rank == kc - 1) bound_key_out[b] = (m == -INFINITY) ? (int)0x80808080 : float_key(m);
}

constexpr int kFinThreads = 256;
constexpr int kMaxCand = 1024;

__global__ void __launch_bounds__(kFinThreads)
finalise_kernel(FinaliseArgs a) {
  __shared__ float s_raw[kMaxCand];
  __shared__ float s_key[kMaxCand];
  __shared__ int64_t s_id[kMaxCand];
  __shared__ uint8_t s_lv[kMaxCand];
  __shared__ float t_raw[ICD_MAX_K];
  __shared__ float t_key[ICD_MAX_K];
  __shared__ double t_w[ICD_MAX_K];
  constexpr int kRed = 8;
  __shared__ double s_red[kRed][kFinThreads / 32];
  __shared__ int s_certified;
  __shared__ int64_t t_id[ICD_MAX_K];
  __shared__ uint8_t t_lv[ICD_MAX_K];
  // cb: this CTA's row of the candidate arrays; b: its query (they differ in the exact fallback's finalise)
  const int cb = blockIdx.x;
  int b = blockIdx.x;
  if (a.fb_in) {
    if (cb >= a.fb_in[0]) return;
    b = a.fb_in[2 + cb];
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kc = a.S * a.kcp;

  // 0. fused exchange, consumer side: the blocks of query b pushed by every peer must have landed
  if (a.wait_flag) {
    if (threadIdx.x < a.S) {
      const uint32_t* f = a.src_stride_bytes
                              ? reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(a.wait_flag) +
                                                                  (size_t)threadIdx.x * a.src_stride_bytes) + b
                              : a.wait_flag + (size_t)threadIdx.x * a.B + b;
      uint32_t spins = 0;
      while (true) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if (v == a.epoch) break;
        if (++spins > (1u << 26)) {
          printf("icdrag: peer flag wait timed out (query %d source %d: have %u want %u)\n", b, threadIdx.x, v, a.epoch);
          __trap();
        }
        __nanosleep(64);
      }
    }
    __syncthreads();
  }

  // 1. gather candidates (ids, scan scores, levels: one parallel round of loads), then exact rescoring -- a warp per
  //    candidate, its row address already in shared memory (id -> row -> dot in one warp cost two dependent L2 round
  //    trips per candidate, nine candidates per warp in a row: 27 - 40 us per launch at small batches, r02w)
  for (int c = threadIdx.x; c < kc; c += kFinThreads) {
    const int s = c / a.kcp, j = c % a.kcp;
    size_t src = ((size_t)s * a.B + cb) * a.kcp + j;
    const float* cs = a.cand_score;
    const int64_t* ci = a.cand_id;
    const uint8_t* cl = a.cand_level;
    if (a.src_stride_bytes) {
      src = (size_t)cb * a.kcp + j;
      cs = reinterpret_cast<const float*>(reinterpret_cast<const char*>(cs) + (size_t)s * a.src_stride_bytes);
      ci = reinterpret_cast<const int64_t*>(reinterpret_cast<const char*>(ci) + (size_t)s * a.src_stride_bytes);
      if (cl) cl += (size_t)s * a.src_stride_bytes;
    }
    const int64_t id = ci[src];
    float raw = cs[src];
    uint8_t lv = 0;
    if (id >= 0) {
      const int64_t local = id - a.row_offset;
      const bool is_local = local >= 0 && local < a.n_local;
      if (cl)
        lv = cl[src];
      else if (is_local && a.levels)
        lv = a.levels[local];
    } else {
      raw = -INFINITY;
    }
    s_raw[c] = raw;
    s_id[c] = id;
    s_lv[c] = lv;
  }
  __syncthreads();
  if (a.q_f32) {
    for (int c = warp; c < kc; c += kFinThreads / 32) {
      const int64_t local = s_id[c] - a.row_offset;
      if (s_id[c] >= 0 && local >= 0 && local < a.n_local) {
        const float raw = a.f32rows ? warp_dot_row<true>(a.rows, local, a.dim, a.q_f32 + (size_t)b * a.dim, lane)
                                    : warp_dot_row<false>(a.rows, local, a.dim, a.q_f32 + (size_t)b * a.dim, lane);
        if (lane == 0) s_raw[c] = raw;
      }
    }
    __syncthreads();
  }
  for (int c = threadIdx.x; c < kc; c += kFinThreads)
    s_key[c] = (a.weight_mode == ICD_WEIGHT_PRE && s_id[c] >= 0) ? s_raw[c] * level_weight_f(s_lv[c]) : s_raw[c];
  __syncthreads();

  // 2. rank sort by (key desc, id asc); empties (id < 0) last; cut to k
  for (int c = threadIdx.x; c < kc; c += kFinThreads) {
    const float kc_s = s_key[c];
    const int64_t kc_i = s_id[c];
    int rank = 0;
    for (int o = 0; o < kc; ++o) {
      if (o == c) continue;
      const float os = s_key[o];
      const int64_t oi = s_id[o];
      bool before;
      if (oi < 0 || kc_i < 0)
        before = (oi >= 0 && kc_i < 0) || (oi < 0 && kc_i < 0 && o < c);
      else
        before = cand_before(os, oi, kc_s, kc_i) || (os == kc_s && oi == kc_i && o < c);
      rank += before ? 1 : 0;
    }
    if (rank < a.k) {
      t_raw[rank] = s_raw[c];
      t_key[rank] = kc_s;
      t_id[rank] = kc_i;
      t_lv[rank] = s_lv[c];
      t_w[rank] = (kc_i < 0) ? -INFINITY
                  : (a.weight_mode == ICD_WEIGHT_RERANK) ? (double)s_raw[c] * level_weight_d(s_lv[c])
                  : (double)kc_s;
    }
  }
  __syncthreads();
  const int kk = min(a.k, kc);

  // 2b. exactness certificate of the tensor path.  Every row outside the candidates has a scan score <= s_kc, the
  //     kc-th candidate's (the scan keeps its top kc, and its pruning bound never exceeds that score).  A row's canonical
  //     score differs from its scan score by at most A (rounding the query to bf16, and the master rows to the bf16
  //     image the scan reads) + T (tensor-core fp32 accumulation, 2 K 2^-24 of the absolute products) + C (the canonical
  //     dot, (L + 5) 2^-24 of them), each bounded per query through the column maxima.  If the k-th returned key beats
  //     s_kc by more than that slack (times the largest level weight under WEIGHT_PRE), no outside row can enter the
  //     top k; otherwise the query is listed for the exact stream scan and writes nothing here.
  if (a.colstat) {
    // each term bounded two ways, through the column maxima and (Cauchy-Schwarz) through the largest row norms
    double r[kRed] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const float* qv = a.q_f32 + (size_t)b * a.dim;
    for (int i = threadIdx.x; i < a.dim; i += kFinThreads) {
      const double qi = qv[i];
      const double bq = (double)__bfloat162float(__float2bfloat16_rn(qv[i]));
      const double M = a.colstat[i], D = a.colstat[a.dim + i];
      r[0] += fabs(qi - bq) * M;
      r[1] += fabs(bq) * D;
      r[2] += fabs(bq) * M;
      r[3] += fabs(qi) * (M + D);
      r[4] += (qi - bq) * (qi - bq);
      r[5] += bq * bq;
      r[6] += qi * qi;
    }
#pragma unroll
    for (int j = 0; j < kRed; ++j) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) r[j] += __shfl_xor_sync(0xffffffffu, r[j], off);
      if (lane == 0) s_red[j][warp] = r[j];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double t[kRed] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
      for (int j = 0; j < kRed; ++j)
        for (int w = 0; w < kFinThreads / 32; ++w) t[j] += s_red[j][w];
      const double R = a.colstat[2 * a.dim], Rd = a.colstat[2 * a.dim + 1];   // max row norms: rows, master - bf16
      const double nd = sqrt(t[4]) * (1.0 + 1e-6), nb = sqrt(t[5]) * (1.0 + 1e-6), nq = sqrt(t[6]) * (1.0 + 1e-6);
      const double A = fmin(t[0], nd * R) + fmin(t[1], nb * Rd);
      const double T = fmin(t[2], nb * R);
      const double Cs = fmin(t[3], nq * (R + Rd));
      const size_t last = (size_t)cb * a.kcp + a.kcp - 1;
      bool ok = true;
      if (a.cand_id[last] >= 0 && kk > 0) {   // a list shorter than kc holds every allowed row
        const double u = 1.0 / 16777216.0;
        const int E = a.f32rows ? 4 : 8;
        const double L = (double)E * ((a.dim + 32 * E - 1) / (32 * E));
        const double slack = A + 2.0 * a.dim * u * T + (L + 5.0) * u * Cs;
        const double wmax = a.weight_mode == ICD_WEIGHT_PRE ? 1.2 : 1.0;
        const double s_kc = a.cand_score[last], kth = t_key[kk - 1];
        ok = kth > s_kc + wmax * slack + 4.0 * u * (fabs(s_kc) + fabs(kth));
      }
      s_certified = ok ? 1 : 0;
      if (!ok) {
        a.fb[2 + atomicAdd(&a.fb[0], 1)] = b;
        atomicAdd(&a.fb[1], 1);
      }
    }
    __syncthreads();
    if (!s_certified) return;
  }

  // 3. reference re-rank: stable sort of the k hits by weighted score, descending
  for (int j = threadIdx.x; j < a.k; j += kFinThreads) {
    size_t dst;
    float o_score, o_raw;
    int64_t o_id;
    uint8_t o_lv;
    if (j < kk) {
      int rank = j;
      if (a.weight_mode == ICD_WEIGHT_RERANK) {
        rank = 0;
        const double w = t_w[j];
        for (int o = 0; o < kk; ++o) rank += (t_w[o] > w || (t_w[o] == w && o < j)) ? 1 : 0;
      }
      dst = (size_t)b * a.k + rank;
      o_score = (float)t_w[j];
      o_raw = t_raw[j];
      o_id = t_id[j];
      o_lv = t_lv[j];
    } else {
      dst = (size_t)b * a.k + j;
      o_score = -INFINITY;
      o_raw = -INFINITY;
      o_id = -1;
      o_lv = 0;
    }
    if (a.out_score) a.out_score[dst] = o_score;
    if (a.out_raw) a.out_raw[dst] = o_raw;
    if (a.out_id) a.out_id[dst] = o_id;
    if (a.out_level) a.out_level[dst] = o_lv;
    for (int pr = 0; pr < a.push.n; ++pr) {
      a.push.raw[pr][dst] = o_raw;
      a.push.id[pr][dst] = o_id;
      a.push.level[pr][dst] = o_lv;
    }
  }
  // fused exchange, producer side: publish this query's block to every peer
  if (a.push.n > 0) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < a.push.n) {
      uint32_t* f = a.push.flag[threadIdx.x] + b;
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(a.push.epoch) : "memory");
    }
  }
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16_rn(in[i]);
}
__global__ void bf16_to_f32_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __bfloat162float(in[i]);
}

// per-column maxima of |value| (bf16 image and master) and of |master - bf16(master)| over a block of rows, folded into
// colstat with integer atomicMax (non-negative floats order like their bit patterns)
constexpr int kStatThreads = 256;
__global__ void __launch_bounds__(kStatThreads)
column_stats_kernel(const __nv_bfloat16* __restrict__ t, const float* __restrict__ m, int64_t n, int dim,
                    float* __restrict__ colstat) {
  constexpr int kCols = 1024 / kStatThreads;
  __shared__ double red[3][kStatThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float mx[kCols], dl[kCols];
#pragma unroll
  for (int j = 0; j < kCols; ++j) mx[j] = dl[j] = 0.f;
  double rmax = 0.0, dmax = 0.0;   // largest squared row norms (thread 0): max(|bf16 row|, |master row|), |master - bf16|
  for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
    double ss_t = 0.0, ss_m = 0.0, ss_d = 0.0;
#pragma unroll
    for (int j = 0; j < kCols; ++j) {
      const int c = threadIdx.x + j * kStatThreads;
      if (c < dim) {
        const float tv = __bfloat162float(t[(size_t)r * dim + c]);
        float av = fabsf(tv);
        ss_t += (double)tv * tv;
        if (m) {
          const float mv = m[(size_t)r * dim + c];
          av = fmaxf(av, fabsf(mv));
          dl[j] = fmaxf(dl[j], fabsf(mv - tv));
          ss_m += (double)mv * mv;
          ss_d += (double)(mv - tv) * (mv - tv);
        }
        mx[j] = fmaxf(mx[j], av);
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      ss_t += __shfl_xor_sync(0xffffffffu, ss_t, off);
      ss_m += __shfl_xor_sync(0xffffffffu, ss_m, off);
      ss_d += __shfl_xor_sync(0xffffffffu, ss_d, off);
    }
    if (lane == 0) red[0][warp] = ss_t, red[1][warp] = ss_m, red[2][warp] = ss_d;
    __syncthreads();
    if (threadIdx.x == 0) {
      double a0 = 0.0, a1 = 0.0, a2 = 0.0;
      for (int w = 0; w < kStatThreads / 32; ++w) a0 += red[0][w], a1 += red[1][w], a2 += red[2][w];
      rmax = fmax(rmax, fmax(a0, a1));
      dmax = fmax(dmax, a2);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    // rounded up: the norms enter an upper bound
    atomicMax(reinterpret_cast<int*>(colstat) + 2 * dim, __float_as_int(__double2float_ru(sqrt(rmax) * (1.0 + 1e-6))));
    atomicMax(reinterpret_cast<int*>(colstat) + 2 * dim + 1, __float_as_int(__double2float_ru(sqrt(dmax) * (1.0 + 1e-6))));
  }
#pragma unroll
  for (int j = 0; j < kCols; ++j) {
    const int c = threadIdx.x + j * kStatThreads;
    if (c < dim) {
      atomicMax(reinterpret_cast<int*>(colstat) + c, __float_as_int(mx[j]));
      atomicMax(reinterpret_cast<int*>(colstat) + dim + c, __float_as_int(dl[j]));
    }
  }
}

}  // namespace

int launch_column_stats(const void* table_bf16, const float* master, int64_t row0, int64_t n, int dim, float* colstat,
                        cudaStream_t st) {
  if (n <= 0) return ICD_OK;
  if (dim > 1024) {
    set_error("column_stats: dim %d > 1024", dim);
    return ICD_E_ARG;
  }
  const int grid = (int)std::min<int64_t>(n, (int64_t)kSMs * 8);
  column_stats_kernel<<<grid, kStatThreads, 0, st>>>(
      reinterpret_cast<const __nv_bfloat16*>(table_bf16) + (size_t)row0 * dim, master ? master + (size_t)row0 * dim : nullptr,
      n, dim, colstat);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

int launch_merge(const MergeArgs& a, cudaStream_t st) {
  if (a.P > kMaxP || a.k_in > 255) {
    set_error("merge: P=%d (max %d) k_in=%d", a.P, kMaxP, a.k_in);
    return ICD_E_ARG;
  }
  const int grid = (a.B + kMergeWarps - 1) / kMergeWarps;
  merge_kernel<<<grid, kMergeWarps * 32, 0, st>>>(a.part_score, a.part_id, a.B, a.P, a.k_in, a.k_out,
                                                 a.out_score, a.out_id, a.row_offset, a.bound_key_out, a.count);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

int launch_bound_from_slots(const float* slot_max, int B, int P, int slots, int kc, int* bound_key_out, cudaStream_t st) {
  if (slots != 32 || kc < 1 || kc > 32 * kFolds || P < 1) {
    set_error("bound_from_slots: slots=%d kc=%d P=%d", slots, kc, P);
    return ICD_E_ARG;
  }
  bound_from_slots_kernel<<<B, kFolds * 32, 0, st>>>(slot_max, B, P, kc, bound_key_out);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

int launch_finalise(const FinaliseArgs& a, cudaStream_t st) {
  if (a.S * a.kcp > kMaxCand || a.k > ICD_MAX_K || a.k < 1) {
    set_error("finalise: S*kcp=%d (max %d), k=%d", a.S * a.kcp, kMaxCand, a.k);
    return ICD_E_ARG;
  }
  finalise_kernel<<<a.B, kFinThreads, 0, st>>>(a);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

int launch_f32_to_bf16(const float* in, void* out, int64_t n, cudaStream_t st) {
  if (n <= 0) return ICD_OK;
  const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)kSMs * 16);
  f32_to_bf16_kernel<<<grid, 256, 0, st>>>(in, reinterpret_cast<__nv_bfloat16*>(out), n);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}
int launch_bf16_to_f32(const void* in, float* out, int64_t n, cudaStream_t st) {
  if (n <= 0) return ICD_OK;
  const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)kSMs * 16);
  bf16_to_f32_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(in), out, n);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

}  // namespace icd
