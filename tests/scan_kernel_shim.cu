// scan_kernel_shim.cu -- test-only extern "C" entries over the scan-side launchers of libicdrag.so.
//
// tests/test_scan_kernels_gpu.py compiles this file into its temporary directory, links it against the shipped
// csrc/libicdrag.so and loads it with ctypes, so the tensor scan, the merge, the pre-pass bound, the finalise certificate
// and the column statistics can each be launched on their own and compared with an fp64 or numpy reference
// (tests/scan_ref.py).  Each entry fills the launch struct from the library header (so its layout cannot drift) and
// returns the launcher's status.  Nothing here allocates, copies or synchronises.  The tensor scan's kernels wait on
// each other through the drift-limiter counters: the Python wrapper, not this file, owns their preconditions.
#include "icdrag.h"
#include "kernels.h"

using namespace icd;

extern "C" {

int shim_tensor_scan(const void* table, const uint8_t* levels, long n_rows, int dim, const void* q_bf16, int B, int k,
                     int weight_pre, float* part_score, int* part_id, int P, int* gbound, int* progress,
                     int tile_stride, int pre_slots, const uint32_t* mask, int* groups_used, void* stream) {
  TensorScanArgs a{};
  a.table = table;
  a.levels = levels;
  a.n_rows = n_rows;
  a.dim = dim;
  a.q_bf16 = q_bf16;
  a.B = B;
  a.k = k;
  a.weight_pre = weight_pre;
  a.part_score = part_score;
  a.part_id = part_id;
  a.P = P;
  a.groups_used = groups_used;
  a.gbound = gbound;
  a.progress = progress;
  a.tile_stride = tile_stride;
  a.pre_slots = pre_slots;
  a.mask = mask;
  // the launcher encodes its own tensor map per launch (the owner argument is unused)
  return launch_tensor_scan(a, nullptr, static_cast<cudaStream_t>(stream));
}

int shim_bound_from_slots(const float* slot_max, int B, int P, int slots, int kc, int* bound_key_out, void* stream) {
  return launch_bound_from_slots(slot_max, B, P, slots, kc, bound_key_out, static_cast<cudaStream_t>(stream));
}

int shim_merge(const float* part_score, const int* part_id, int B, int P, int k_in, int k_out, float* out_score,
               int64_t* out_id, long row_offset, int* bound_key_out, const int* count, void* stream) {
  MergeArgs m{};
  m.part_score = part_score;
  m.part_id = part_id;
  m.B = B;
  m.P = P;
  m.k_in = k_in;
  m.k_out = k_out;
  m.out_score = out_score;
  m.out_id = out_id;
  m.row_offset = row_offset;
  m.bound_key_out = bound_key_out;
  m.count = count;
  return launch_merge(m, static_cast<cudaStream_t>(stream));
}

// local finalise of one shard (S = 1): never waits on flags and pushes nowhere
int shim_finalise(const float* cand_score, const int64_t* cand_id, int B, int kcp, int k, long row_offset,
                  long n_local, const float* q_f32, const void* rows, int f32rows, int dim, const uint8_t* levels,
                  int weight_mode, float* out_score, float* out_raw, int64_t* out_id, uint8_t* out_level,
                  const float* colstat, int* fb, const int* fb_in, void* stream) {
  FinaliseArgs f{};
  f.cand_score = cand_score;
  f.cand_id = cand_id;
  f.S = 1;
  f.B = B;
  f.kcp = kcp;
  f.k = k;
  f.row_offset = row_offset;
  f.n_local = n_local;
  f.q_f32 = q_f32;
  f.rows = rows;
  f.f32rows = f32rows != 0;
  f.dim = dim;
  f.levels = levels;
  f.weight_mode = weight_mode;
  f.out_score = out_score;
  f.out_raw = out_raw;
  f.out_id = out_id;
  f.out_level = out_level;
  f.colstat = colstat;
  f.fb = fb;
  f.fb_in = fb_in;
  return launch_finalise(f, static_cast<cudaStream_t>(stream));
}

int shim_column_stats(const void* table_bf16, const float* master, long row0, long n, int dim, float* colstat,
                      void* stream) {
  return launch_column_stats(table_bf16, master, row0, n, dim, colstat, static_cast<cudaStream_t>(stream));
}

int shim_tensor_scan_sample_stride(long n_rows, int kc) { return tensor_scan_sample_stride(n_rows, kc); }
int shim_tensor_scan_max_partials(void) { return tensor_scan_max_partials(); }
int shim_tensor_scan_pre_slots(void) { return tensor_scan_pre_slots(); }
int shim_tensor_scan_pre_capacity(void) { return tensor_scan_pre_capacity(); }
int shim_tensor_scan_progress_ints(void) { return tensor_scan_progress_ints(); }

}  // extern "C"
