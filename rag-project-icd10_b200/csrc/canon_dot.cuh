// canon_dot.cuh -- the canonical exact fp32 dot of a query with a table row.
//
// Chunk c (16 bytes: 8 bf16 or 4 fp32 elements) of the row belongs to lane c % 32; each lane accumulates its chunks in
// ascending order, elements ascending, with fmaf; then an xor butterfly (16, 8, 4, 2, 1) sums the lanes.  This is the
// order of scan_stream.cu, the order finalise_kernel rescores in, and the order the paged search (topk_large.cu) scores
// every row in, so all of them return bit-identical raw scores.
#pragma once
#include "common.cuh"

namespace icd {

// one 16-byte chunk of the row times the matching query slice qs[0 .. E)
template <bool F32ROWS>
__device__ __forceinline__ float canon_chunk_fma(const uint4& v, const float* qs, float acc) {
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

__device__ __forceinline__ float canon_lane_sum(float acc) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  return acc;
}

// canonical exact dot of row `row` with q (every lane of the warp returns it)
template <bool F32ROWS>
__device__ __forceinline__ float warp_dot_row(const void* rows, int64_t row, int dim, const float* q, int lane) {
  constexpr int E = F32ROWS ? 4 : 8;
  const int nchunks = dim / E;
  const char* base = reinterpret_cast<const char*>(rows) + (size_t)row * dim * (F32ROWS ? 4 : 2);
  float acc = 0.f;
  for (int c = lane; c < nchunks; c += 32) {
    const uint4 v = *reinterpret_cast<const uint4*>(base + (size_t)c * 16);
    acc = canon_chunk_fma<F32ROWS>(v, q + c * E, acc);
  }
  return canon_lane_sum(acc);
}

}  // namespace icd
