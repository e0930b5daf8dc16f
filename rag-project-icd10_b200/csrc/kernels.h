// kernels.h -- host-side launch interfaces between the translation units of libicdrag.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace icd {

// ---- scan_stream.cu
struct StreamScanArgs {
  const void* table;      // [n_rows, dim] bf16 or fp32 (f32rows)
  const uint8_t* levels;  // [n_rows]
  int64_t n_rows;
  int dim;
  bool f32rows;
  const float* q;  // [nq, dim] fp32, first query of this pass
  int nq;          // queries in this pass (<= stream_scan_max_queries)
  int q0;          // index of the first query of this pass within the batch (partial buffer row)
  int k;
  int weight_pre;
  float* part_score;  // [B, P, k]
  int* part_id;       // [B, P, k] local row, -1 = empty
  int P;              // partial lists per query == grid size
  const uint32_t* mask;  // row bitmap (bit i & 31 of word i >> 5 = row i may be returned), null = every row
};
int stream_scan_grid();
int stream_scan_max_queries(bool f32rows, int dim);
int launch_stream_scan(const StreamScanArgs& a, cudaStream_t st);
// exact fallback of the tensor path: one query per pass over the queries listed in device memory (fb = [count, total,
// query ids...] as finalise_kernel leaves it); a.q is the whole batch [B, dim], a.nq = B bounds the list, slot j of the
// list writes partial row j.  The count stays on the device, so the call does not synchronise.
int launch_stream_scan_listed(const StreamScanArgs& a, const int* fb, cudaStream_t st);

// ---- scan_tc.cu (tcgen05 / TMEM / TMA)
struct TensorScanArgs {
  const void* table;      // [n_rows, dim] bf16, 16-byte aligned rows
  const uint8_t* levels;  // [n_rows]
  int64_t n_rows;
  int dim;                 // multiple of 64, <= 768
  const void* q_bf16;      // [B, dim] bf16 device
  int B;
  int k;
  int weight_pre;
  float* part_score;  // [B, P, k]
  int* part_id;       // [B, P, k]
  int P;              // partial lists per query the buffers were sized for (>= groups used)
  int* groups_used;   // out: partial lists actually written per query
  int* gbound;        // [B] ints, pre-set to 0x80808080 (a very negative key), or null to disable pruning
  int* progress;      // [tensor_scan_progress_ints()] zeroed ints for the drift limiter, or null
  int tile_stride;    // 0/1: scan every row; s > 1: scan every s-th 128-row tile only (sampling pre-pass)
  int pre_slots;      // != 0 (with tile_stride > 1): slot-maxima pre-pass -- part_score receives [B, groups, tensor_scan_pre_slots()]
                      // running maxima instead of sorted lists, part_id is untouched; feed launch_bound_from_slots
  const uint32_t* mask;  // row bitmap as StreamScanArgs::mask, null = every row
};
int tensor_scan_pre_slots();
int tensor_scan_pre_capacity();   // largest kc the slot-maxima bound serves (slots x the row-group classes it keeps apart)
int tensor_scan_pre_mode();   // 1 = slot-maxima pre-pass (default), 0 = list-based pre-pass (icd_tune "scan_pre_slots")
// stride of the sampling pre-pass for a table of n_rows when the scan keeps kc candidates per query (0 = no pre-pass)
int tensor_scan_sample_stride(int64_t n_rows, int kc);
// run-time tuning (icd_tune); the generation moves whenever a knob that shapes the TMA descriptor changes
int tensor_scan_tune(const char* key, int value);
int tensor_scan_generation();
int tensor_scan_max_partials();
int tensor_scan_progress_ints();
bool tensor_scan_supported(int dim, int k);
int launch_tensor_scan(const TensorScanArgs& a, const void* tensor_map_owner, cudaStream_t st);
// builds (or rebuilds) the TMA descriptor of the table; owner is an opaque 128-byte aligned blob
int tensor_scan_make_map(void* map128, const void* table, int64_t n_rows, int dim);

// ---- topk_merge.cu
struct MergeArgs {
  const float* part_score;  // [B, P, k_in] each list sorted (score desc, id asc); -inf/-1 padded
  const int* part_id;       // [B, P, k_in] local rows
  int B, P, k_in;
  int k_out;                 // <= k_in
  float* out_score;          // [B, k_out]
  int64_t* out_id;           // [B, k_out] local row + row_offset, -1 = empty
  int64_t row_offset;
  int* bound_key_out;        // [B] or null: order-preserving key of the k_out-th score (very negative when
                             // the list holds fewer than k_out rows) -- the admission bound of the main scan
  const int* count;          // or null: only the first *count of the B lists are live (the exact fallback's)
};
int launch_merge(const MergeArgs& a, cudaStream_t st);
// pre-pass bound: per query the kc-th largest of the slot maxima (each slot's maximum taken over the row groups of one
// class g mod 4) as an order-preserving key in bound_key_out[b]; slots is tensor_scan_pre_slots() (32),
// kc <= tensor_scan_pre_capacity() (128)
int launch_bound_from_slots(const float* slot_max /*[B, P, slots]*/, int B, int P, int slots, int kc, int* bound_key_out,
                            cudaStream_t st);

// fused exchange, producer side: per-peer destinations of this rank's (raw, id, level) block
struct PushTargets {
  int n;
  float* raw[8];
  int64_t* id[8];
  uint8_t* level[8];
  uint32_t* flag[8];  // [B] per peer; flag[b] = epoch published with system-scope release
  uint32_t epoch;
};

struct FinaliseArgs {
  // candidate lists from S sources (S = 1 locally, S = world after a shard exchange),
  // laid out [S][B][kcp]; total S*kcp <= 1024
  const float* cand_score;
  const int64_t* cand_id;       // global ids, -1 = empty
  const uint8_t* cand_level;    // [S][B][kcp] or null -> levels[id - row_offset]
  size_t src_stride_bytes;      // 0: arrays are dense [S][B][kcp]; else source s starts s*stride bytes later
  int S, B, kcp, k;
  int64_t row_offset;  // global id - row_offset = local row
  int64_t n_local;
  // exact rescoring (optional: q_f32 == nullptr keeps cand_score). Canonical fp32 order of
  // scan_stream.cu so both scan paths return bit-identical scores.
  const float* q_f32;  // [B, dim]
  const void* rows;    // bf16 table or fp32 master of the local shard
  bool f32rows;
  int dim;
  const uint8_t* levels;  // local levels
  int weight_mode;        // ICD_WEIGHT_*
  float* out_score;    // [B, k] may be null
  float* out_raw;      // [B, k] may be null
  int64_t* out_id;     // [B, k] may be null
  uint8_t* out_level;  // [B, k] may be null
  // fused exchange, producer side: after its [k] block is written, CTA b also stores the
  // (raw, id, level) block into every peer's receive slab over NVLink-mapped pointers and
  // publishes flag[b] = epoch there (system-scope release).
  PushTargets push;
  // fused exchange, consumer side: CTA b waits for wait_flag[s][b] == epoch of every source
  const uint32_t* wait_flag;  // [S][B] or null
  uint32_t epoch;
  // Exactness certificate of the tensor path (colstat != null, S == 1): cand_score holds the scan's own scores, and a
  // query is certified when its k-th canonical key beats the kc-th scan score by more than the scan's error bound
  // (DESIGN.md, "Exact search").  An uncertified query writes nothing and appends its id to fb = [count, total, ids...].
  const float* colstat;  // [2][dim]: max |row_i| (bf16 image and master), max |master_i - bf16(master_i)|; then the
                         // largest row norm (either copy) and the largest |master row - bf16 row|
  int* fb;
  // the fallback's finalise: CTA j serves query fb_in[2 + j] if j < fb_in[0], its candidates in row j of cand_*
  const int* fb_in;
};
int launch_finalise(const FinaliseArgs& a, cudaStream_t st);

// ---- topk_large.cu: exact paged search, K = offset + limit <= ICD_MAX_LIMIT (icd_index_search_page)
struct PageSearchArgs {
  const void* rows;       // [n, dim] bf16 table or fp32 master (f32rows): the rows finalise_kernel rescores
  bool f32rows;
  const uint8_t* levels;  // [n]
  int64_t n;
  int dim;
  const float* q;         // [nq, dim] fp32 device
  int nq;
  const uint32_t* mask;   // row bitmap, null = every row
  int range_flags;        // ICD_RANGE_RADIUS | ICD_RANGE_FILTER, on the raw inner product
  float radius, range_filter;
  int weight_mode;
  int offset, limit;
  int chunk;              // queries per workspace pass (page_search_chunk)
  void* workspace;        // page_search_workspace_bytes(n, offset + limit, chunk) device bytes
  size_t workspace_bytes;
  float* out_score;       // [nq, limit] device, each may be null
  float* out_raw;
  int64_t* out_id;
};
// queries per pass for a batch of B: the [chunk, n] fp32 score workspace stays within a fixed budget (512 MiB)
int page_search_chunk(int64_t n, int K, int B);
size_t page_search_workspace_bytes(int64_t n, int K, int chunk);
int launch_page_search(const PageSearchArgs& a, cudaStream_t st);

// elementwise helpers
int launch_f32_to_bf16(const float* in, void* out_bf16, int64_t n, cudaStream_t st);
int launch_bf16_to_f32(const void* in_bf16, float* out, int64_t n, cudaStream_t st);
// per-column maxima of rows [row0, row0 + n) folded into colstat (see FinaliseArgs::colstat); master may be null
int launch_column_stats(const void* table_bf16, const float* master, int64_t row0, int64_t n, int dim, float* colstat,
                        cudaStream_t st);

}  // namespace icd
