// scan_stream.cu -- HBM-stream exact inner-product scan with fused top-k (small query batches).
//
// Replaces the brute-force FLAT/IP search inside MilvusClient.search
// (reference call site services/milvus_service.py:280-285) for 1..4 queries per pass:
// every table row is read exactly once with coalesced 128-bit loads, all queries of the
// pass are scored against it in fp32 (products of bf16/fp32 values, fp32 FMA accumulate in a
// fixed order), and a per-warp sorted list keeps the running top-k, so the [B, N] score
// matrix never exists.  Per-CTA lists go to a partial buffer that topk_merge.cu reduces.
//
// Roofline: HBM.  Algorithmic bytes per row = dim*2 (+1 level byte when weighting before
// selection); see DESIGN.md section "Kernels".
#include "common.cuh"
#include "kernels.h"

namespace icd {

namespace {

constexpr int kWarps = 8;  // warps per CTA

template <bool F32ROWS>
struct RowChunk {
  // number of elements in one 16-byte chunk
  static constexpr int kElems = F32ROWS ? 4 : 8;
};

// Dot of one 16-byte chunk with the matching query slice, accumulated in canonical order.
template <bool F32ROWS>
__device__ __forceinline__ float chunk_fma(const uint4& v, const float* qs, float acc) {
  if constexpr (F32ROWS) {
    acc = fmaf(__uint_as_float(v.x), qs[0], acc);
    acc = fmaf(__uint_as_float(v.y), qs[1], acc);
    acc = fmaf(__uint_as_float(v.z), qs[2], acc);
    acc = fmaf(__uint_as_float(v.w), qs[3], acc);
  } else {
    acc = fmaf(bf16lo_to_f32(v.x), qs[0], acc);
    acc = fmaf(bf16hi_to_f32(v.x), qs[1], acc);
    acc = fmaf(bf16lo_to_f32(v.y), qs[2], acc);
    acc = fmaf(bf16hi_to_f32(v.y), qs[3], acc);
    acc = fmaf(bf16lo_to_f32(v.z), qs[4], acc);
    acc = fmaf(bf16hi_to_f32(v.z), qs[5], acc);
    acc = fmaf(bf16lo_to_f32(v.w), qs[6], acc);
    acc = fmaf(bf16hi_to_f32(v.w), qs[7], acc);
  }
  return acc;
}

__device__ __forceinline__ float warp_sum_all(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// Warp-cooperative insert of (s, id) into a sorted list of k entries held in shared memory.
// Returns the new k-th score (the admission threshold).
__device__ __forceinline__ float warp_list_insert(float* sc, int* id, int k, float s, int rid, int lane) {
  int cnt = 0;
  for (int e = lane; e < k; e += 32) cnt += cand_before(sc[e], id[e], s, rid) ? 1 : 0;
  const int pos = __reduce_add_sync(0xffffffffu, cnt);
  // shift [pos, k-2] -> [pos+1, k-1]
  float ts[ICD_MAX_K / 32];
  int ti[ICD_MAX_K / 32];
#pragma unroll
  for (int j = 0; j < ICD_MAX_K / 32; ++j) {
    const int e = lane + 32 * j;
    if (e > pos && e < k) {
      ts[j] = sc[e - 1];
      ti[j] = id[e - 1];
    }
  }
  __syncwarp();
#pragma unroll
  for (int j = 0; j < ICD_MAX_K / 32; ++j) {
    const int e = lane + 32 * j;
    if (e > pos && e < k) {
      sc[e] = ts[j];
      id[e] = ti[j];
    }
  }
  if (lane == 0 && pos < k) {
    sc[pos] = s;
    id[pos] = rid;
  }
  __syncwarp();
  return sc[k - 1];
}

// NQ queries per pass, CPL 16-byte chunks per lane per row, R rows in flight per warp.  MASKED: only rows whose bit is
// set in `mask` are read and inserted (a template parameter: the widest variants have no register to spare, so the
// unfiltered scan stays exactly what it was).
template <int NQ, int CPL, bool F32ROWS, int R, bool MASKED>
__device__ __forceinline__ void scan_stream_body(const void* __restrict__ table, const uint8_t* __restrict__ levels,
                                                 int64_t n_rows, int dim, const float* __restrict__ q, int nq_valid,
                                                 int k, int weight_pre, float* __restrict__ part_score,
                                                 int* __restrict__ part_id, int q0, int P,
                                                 const uint32_t* __restrict__ mask) {
  constexpr int E = RowChunk<F32ROWS>::kElems;
  constexpr int kRowsPerWarpIter = R;
  constexpr int kRowsPerCtaIter = kWarps * R;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunks = dim / E;
  const size_t row_bytes = (size_t)dim * (F32ROWS ? 4 : 2);

  // per-warp, per-query sorted lists
  float* lists_s = reinterpret_cast<float*>(smem_raw);                     // [kWarps][NQ][k]
  int* lists_i = reinterpret_cast<int*>(lists_s + kWarps * NQ * k);        // [kWarps][NQ][k]
  float* my_s = lists_s + (size_t)warp * NQ * k;
  int* my_i = lists_i + (size_t)warp * NQ * k;
  for (int e = lane; e < NQ * k; e += 32) {
    my_s[e] = -INFINITY;
    my_i[e] = 0x7fffffff;
  }
  __syncwarp();

  // query slices owned by this lane: chunk c = lane + 32*i
  float qreg[NQ][CPL * E];
#pragma unroll
  for (int b = 0; b < NQ; ++b) {
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = lane + 32 * i;
#pragma unroll
      for (int e = 0; e < E; ++e)
        qreg[b][i * E + e] = (c < nchunks && b < nq_valid) ? q[(size_t)b * dim + c * E + e] : 0.f;
    }
  }

  float thr[NQ];
#pragma unroll
  for (int b = 0; b < NQ; ++b) thr[b] = -INFINITY;

  // Row mask: the R rows of a warp step lie in one mask word (R divides 32 and wrow is a multiple of R).  The word of
  // the next step is loaded one step ahead, so its L2 round trip does not stand in front of the row loads.
  auto mask_bits = [&](int64_t wrow) -> uint32_t {
    if constexpr (!MASKED) return 0xffffffffu;
    return wrow < n_rows ? __ldg(mask + (wrow >> 5)) >> (wrow & 31) : 0u;
  };
  const char* base = reinterpret_cast<const char*>(table);
  uint32_t next_bits = mask_bits((int64_t)blockIdx.x * kRowsPerCtaIter + warp * kRowsPerWarpIter);
  for (int64_t row0 = (int64_t)blockIdx.x * kRowsPerCtaIter; row0 < n_rows;
       row0 += (int64_t)gridDim.x * kRowsPerCtaIter) {
    const int64_t wrow = row0 + warp * kRowsPerWarpIter;
    const uint32_t bits = next_bits;
    if constexpr (MASKED) next_bits = mask_bits(wrow + (int64_t)gridDim.x * kRowsPerCtaIter);
    uint4 v[kRowsPerWarpIter][CPL];
#pragma unroll
    for (int r = 0; r < kRowsPerWarpIter; ++r) {
      const int64_t row = wrow + r;
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = lane + 32 * i;
        if (row < n_rows && c < nchunks && (!MASKED || ((bits >> r) & 1u)))
          v[r][i] = ld_stream_u4(base + (size_t)row * row_bytes + (size_t)c * 16);
        else
          v[r][i] = make_uint4(0, 0, 0, 0);
      }
    }
#pragma unroll
    for (int r = 0; r < kRowsPerWarpIter; ++r) {
      const int64_t row = wrow + r;
      if (row >= n_rows) break;  // warp-uniform
      if (MASKED && !((bits >> r) & 1u)) continue;
      float acc[NQ];
#pragma unroll
      for (int b = 0; b < NQ; ++b) acc[b] = 0.f;
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
#pragma unroll
        for (int b = 0; b < NQ; ++b) acc[b] = chunk_fma<F32ROWS>(v[r][i], &qreg[b][i * E], acc[b]);
      }
      float w = 1.f;
      if (weight_pre) w = level_weight_f(levels[row]);
#pragma unroll
      for (int b = 0; b < NQ; ++b) {
        float s = warp_sum_all(acc[b]);
        if (weight_pre) s *= w;
        if (b < nq_valid && s > thr[b])  // warp-uniform: every lane holds the same s
          thr[b] = warp_list_insert(my_s + b * k, my_i + b * k, k, s, (int)row, lane);
      }
    }
  }
  __syncthreads();

  // CTA merge: warp b (b < NQ) merges the kWarps lists of query b by repeated head selection
  if (warp < NQ && warp < nq_valid) {
    const int b = warp;
    int head = 0;  // lanes 0..kWarps-1 each walk one list
    float* out_s = part_score + ((size_t)(q0 + b) * P + blockIdx.x) * k;
    int* out_i = part_id + ((size_t)(q0 + b) * P + blockIdx.x) * k;
    for (int j = 0; j < k; ++j) {
      float s = -INFINITY;
      int id = 0x7fffffff;
      if (lane < kWarps && head < k) {
        s = lists_s[((size_t)lane * NQ + b) * k + head];
        id = lists_i[((size_t)lane * NQ + b) * k + head];
      }
      // warp argbest over (s, id)
      float bs = s;
      int bi = id, bl = lane;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const float os = __shfl_xor_sync(0xffffffffu, bs, off);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
        const int ol = __shfl_xor_sync(0xffffffffu, bl, off);
        if (cand_before(os, oi, bs, bi) || (os == bs && oi == bi && ol < bl)) {
          bs = os;
          bi = oi;
          bl = ol;
        }
      }
      if (lane == bl) ++head;
      if (lane == 0) {
        out_s[j] = bs;
        out_i[j] = (bs == -INFINITY) ? -1 : bi;
      }
    }
  }
}

template <int NQ, int CPL, bool F32ROWS, int R, bool MASKED>
__global__ void __launch_bounds__(kWarps * 32, 2)
scan_stream_kernel(const void* __restrict__ table, const uint8_t* __restrict__ levels, int64_t n_rows,
                   int dim, const float* __restrict__ q, int nq_valid, int k, int weight_pre,
                   float* __restrict__ part_score, int* __restrict__ part_id, int q0, int P,
                   const uint32_t* __restrict__ mask) {
  scan_stream_body<NQ, CPL, F32ROWS, R, MASKED>(table, levels, n_rows, dim, q, nq_valid, k, weight_pre, part_score,
                                                part_id, q0, P, mask);
}

// The tensor path's exact fallback: the queries listed in fb[2 ..] (fb[0] of them, at most nq_max), one per pass; grid.y
// slots walk the list, slot j's partial lists go to row j of the partial buffer.
template <int CPL, bool F32ROWS, int R, bool MASKED>
__global__ void __launch_bounds__(kWarps * 32, 2)
scan_stream_listed_kernel(const void* __restrict__ table, const uint8_t* __restrict__ levels, int64_t n_rows,
                          int dim, const float* __restrict__ q, int nq_max, int k, int weight_pre,
                          float* __restrict__ part_score, int* __restrict__ part_id, int P,
                          const uint32_t* __restrict__ mask, const int* __restrict__ fb) {
  const int count = min(fb[0], nq_max);
  for (int j = blockIdx.y; j < count; j += gridDim.y) {
    const float* qj = q + (size_t)fb[2 + j] * dim;
    scan_stream_body<1, CPL, F32ROWS, R, MASKED>(table, levels, n_rows, dim, qj, 1, k, weight_pre, part_score, part_id,
                                                 j, P, mask);
    __syncthreads();   // the next pass re-initialises the lists this pass's merge reads
  }
}

template <int NQ, int CPL, bool F32ROWS, int R>
int launch_one(const StreamScanArgs& a, int grid, size_t smem, cudaStream_t st) {
  auto kern = a.mask ? scan_stream_kernel<NQ, CPL, F32ROWS, R, true> : scan_stream_kernel<NQ, CPL, F32ROWS, R, false>;
  ICD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kWarps * 32, smem, st>>>(a.table, a.levels, a.n_rows, a.dim, a.q, a.nq, a.k,
                                        a.weight_pre, a.part_score, a.part_id, a.q0, a.P, a.mask);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

// bf16 rows: up to 4 chunks per lane (dim <= 1024); 4 rows in flight for 1-2 queries, 2 for 4
template <int NQ>
int launch_bf16(const StreamScanArgs& a, int grid, size_t smem, cudaStream_t st) {
  constexpr int R = NQ >= 4 ? 2 : 4;
  const int cpl = (a.dim / 8 + 31) / 32;
  switch (cpl) {
    case 1: return launch_one<NQ, 1, false, R>(a, grid, smem, st);
    case 2: return launch_one<NQ, 2, false, R>(a, grid, smem, st);
    case 3: return launch_one<NQ, 3, false, R>(a, grid, smem, st);
    case 4:
      if constexpr (NQ <= 2) return launch_one<NQ, 4, false, R>(a, grid, smem, st);
      break;
    default: break;
  }
  set_error("scan_stream: dim %d not supported with %d queries per pass", a.dim, NQ);
  return ICD_E_UNSUPPORTED;
}

// fp32 master rows: up to 8 chunks per lane (dim <= 1024), 2 rows in flight, one query per pass
int launch_f32(const StreamScanArgs& a, int grid, size_t smem, cudaStream_t st) {
  const int cpl = (a.dim / 4 + 31) / 32;
  switch (cpl) {
    case 1: return launch_one<1, 1, true, 4>(a, grid, smem, st);
    case 2: return launch_one<1, 2, true, 4>(a, grid, smem, st);
    case 3: return launch_one<1, 3, true, 2>(a, grid, smem, st);
    case 4: return launch_one<1, 4, true, 2>(a, grid, smem, st);
    case 5:
    case 6: return launch_one<1, 6, true, 2>(a, grid, smem, st);
    case 7:
    case 8: return launch_one<1, 8, true, 2>(a, grid, smem, st);
    default: break;
  }
  set_error("scan_stream: dim %d not supported (fp32 rows need dim %% 4 == 0, dim <= 1024)", a.dim);
  return ICD_E_UNSUPPORTED;
}

template <int CPL, bool F32ROWS, int R>
int launch_listed_one(const StreamScanArgs& a, const int* fb, size_t smem, cudaStream_t st) {
  auto kern = a.mask ? scan_stream_listed_kernel<CPL, F32ROWS, R, true> : scan_stream_listed_kernel<CPL, F32ROWS, R, false>;
  ICD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // 8 list slots in flight: a handful of uncertified queries costs one pass over the table, and a CTA whose slots are
  // past the count exits at once
  const dim3 grid(a.P, std::min(a.nq, 8));
  kern<<<grid, kWarps * 32, smem, st>>>(a.table, a.levels, a.n_rows, a.dim, a.q, a.nq, a.k, a.weight_pre, a.part_score,
                                        a.part_id, a.P, a.mask, fb);
  count_launch();
  ICD_CUDA(cudaGetLastError());
  return ICD_OK;
}

}  // namespace

int launch_stream_scan_listed(const StreamScanArgs& a, const int* fb, cudaStream_t st) {
  const size_t smem = (size_t)kWarps * a.k * 8;
  if (a.f32rows) {
    switch ((a.dim / 4 + 31) / 32) {
      case 1: return launch_listed_one<1, true, 4>(a, fb, smem, st);
      case 2: return launch_listed_one<2, true, 4>(a, fb, smem, st);
      case 3: return launch_listed_one<3, true, 2>(a, fb, smem, st);
      case 4: return launch_listed_one<4, true, 2>(a, fb, smem, st);
      case 5:
      case 6: return launch_listed_one<6, true, 2>(a, fb, smem, st);
      default: break;
    }
  } else {
    switch ((a.dim / 8 + 31) / 32) {
      case 1: return launch_listed_one<1, false, 4>(a, fb, smem, st);
      case 2: return launch_listed_one<2, false, 4>(a, fb, smem, st);
      case 3: return launch_listed_one<3, false, 4>(a, fb, smem, st);
      default: break;
    }
  }
  set_error("scan_stream: no listed variant for dim %d (the tensor path serves dim <= 768)", a.dim);
  return ICD_E_UNSUPPORTED;
}

int stream_scan_grid() { return kSMs * 2; }
int stream_scan_max_queries(bool f32rows, int dim) { return f32rows ? 1 : (dim > 768 ? 2 : 4); }

int launch_stream_scan(const StreamScanArgs& a, cudaStream_t st) {
  const int grid = a.P;
  if (a.f32rows) {
    if (a.nq != 1) {
      set_error("scan_stream: fp32 rows take one query per pass");
      return ICD_E_ARG;
    }
    return launch_f32(a, grid, (size_t)kWarps * a.k * 8, st);
  }
  const int nqt = a.nq <= 1 ? 1 : (a.nq <= 2 ? 2 : 4);
  const size_t smem = (size_t)kWarps * nqt * a.k * 8;
  if (nqt == 1) return launch_bf16<1>(a, grid, smem, st);
  if (nqt == 2) return launch_bf16<2>(a, grid, smem, st);
  return launch_bf16<4>(a, grid, smem, st);
}

}  // namespace icd
