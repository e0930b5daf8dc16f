// index_impl.h -- private layout of the opaque icd_index handle.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/icdrag.h"
#include "kernels.h"

namespace icd {

struct DeviceBuf {
  void* ptr = nullptr;
  size_t cap = 0;
  int reserve(size_t bytes);
  void release();
};

}  // namespace icd

struct icd_index {
  int dim = 0, device = 0, flags = 0;
  int64_t cap = 0, n = 0;
  bool adopted = false;
  // HBM layout: row-major [n, dim] bf16 table (the scanned copy), optional fp32 master,
  // one level byte per row
  void* table = nullptr;
  float* master = nullptr;
  uint8_t* levels = nullptr;
  // TMA descriptor of `table` for the tensor scan (CUtensorMap is 128 bytes, 64-byte aligned)
  alignas(128) unsigned char tmap[128];
  bool map_valid = false;
  int64_t map_rows = 0;
  int map_gen = -1;
  // workspace
  icd::DeviceBuf q_f32, q_bf16, part_score, part_id, cand_score, cand_id, out_stage, in_stage, gbound;
  icd::DeviceBuf mask;   // a row mask handed over in host memory, copied in like the queries
  // exactness certificate of the tensor path: [2][dim] column maxima and 2 row-norm maxima (launch_column_stats), the list of
  // queries it could not certify: [count of this search, total since icd_index_take_fallbacks, query ids (<= 8192)]
  icd::DeviceBuf colstat, fb;
  // pipelined searches from host buffers (icd_index_search, large batches): the second set of query / result staging
  // buffers, the copy stream and the events that order the two streams
  icd::DeviceBuf q_f32_alt, q_bf16_alt, out_stage_alt;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};   // [set]: copied in / searched
  // stage timing (scan, merge, finalise): a ring of event quads so that back-to-back searches can be averaged
  // afterwards without a host sync between them (bench.py's roofline figure); ev = the quad of the current call
  static constexpr int kTimingRing = 64;
  cudaEvent_t ev_ring[kTimingRing][4];
  cudaEvent_t* ev = ev_ring[0];
  int64_t timed_calls = 0;   // searches recorded since timing was switched on
  bool timing = false, timing_pending = false;
  int last_launches = 0;
  icd::DeviceBuf page_ws;   // icd_index_search_page: [chunk, n] scores, select state, gathered lists (topk_large.cu)
};

namespace icd {
int index_stage_queries(icd_index* x, const void* q, int q_dtype, int B, cudaStream_t st);
int index_search_device(icd_index* x, int B, int k, int weight_mode, int path, int64_t row_offset,
                        float* d_score, float* d_raw, int64_t* d_id, uint8_t* d_level,
                        bool q_exact_bf16, const PushTargets* push, const uint32_t* d_mask, cudaStream_t st);
// row mask of a filtered search: checks mask_rows == x->n, copies a host mask into the workspace; *d_mask = the device
// mask, or null when row_mask is null (every row)
int index_stage_mask(icd_index* x, const uint32_t* row_mask, int64_t mask_rows, const uint32_t** d_mask, cudaStream_t st);
int copy_out(void* dst, const void* src_dev, size_t bytes, cudaStream_t st);
}  // namespace icd
