// api_index.cu -- the C ABI of the vector table: append / search orchestration.
//
// Stands where MilvusClient.insert / MilvusClient.search stand in the reference
// (services/milvus_service.py:259,280-285).  Kernels live in scan_stream.cu, scan_tc.cu and
// topk_merge.cu; this file owns the device buffers, picks the scan path and stages host
// buffers.
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "index_impl.h"
#include "kernels.h"
#include "encoder_kernels.h"

namespace icd {

static thread_local std::string t_error;
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  t_error = buf;
}

int DeviceBuf::reserve(size_t bytes) {
  if (bytes <= cap) return ICD_OK;
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
  ICD_CUDA(cudaMalloc(&ptr, bytes));
  cap = bytes;
  return ICD_OK;
}
void DeviceBuf::release() {
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

static int alloc_table(icd_index* x, int64_t cap) {
  const size_t row_bf16 = (size_t)x->dim * 2;
  void* t = nullptr;
  float* m = nullptr;
  uint8_t* l = nullptr;
  ICD_CUDA(cudaMalloc(&t, std::max<size_t>(row_bf16 * cap, 256)));
  if (x->flags & ICD_INDEX_KEEP_F32) ICD_CUDA(cudaMalloc(&m, std::max<size_t>((size_t)x->dim * 4 * cap, 256)));
  ICD_CUDA(cudaMalloc(&l, std::max<size_t>(cap, 256)));
  if (x->n > 0) {
    ICD_CUDA(cudaMemcpy(t, x->table, row_bf16 * x->n, cudaMemcpyDeviceToDevice));
    if (m) ICD_CUDA(cudaMemcpy(m, x->master, (size_t)x->dim * 4 * x->n, cudaMemcpyDeviceToDevice));
    ICD_CUDA(cudaMemcpy(l, x->levels, x->n, cudaMemcpyDeviceToDevice));
  }
  if (x->table) cudaFree(x->table);
  if (x->master) cudaFree(x->master);
  if (x->levels) cudaFree(x->levels);
  x->table = t;
  x->master = m;
  x->levels = l;
  x->cap = cap;
  x->map_valid = false;
  return ICD_OK;
}

// ------------------------------------------------------------------------------------------
// local search on device buffers: q_f32 / q_bf16 already staged in the workspace.
// Writes [B, k] results into the given DEVICE buffers (any may be null).
int index_search_device(icd_index* x, int B, int k, int weight_mode, int path, int64_t row_offset,
                        float* d_score, float* d_raw, int64_t* d_id, uint8_t* d_level,
                        bool q_exact_bf16, const PushTargets* push, const uint32_t* d_mask, cudaStream_t st) {
  const int64_t n = x->n;
  const bool have_master = x->master != nullptr;
  const int weight_pre = weight_mode == ICD_WEIGHT_PRE ? 1 : 0;
  // path choice
  bool use_tc = false;
  if (path == ICD_PATH_TENSOR) {
    if (!tensor_scan_supported(x->dim, k)) {
      set_error("tensor scan needs dim %% 64 == 0, dim <= 768 (dim=%d)", x->dim);
      return ICD_E_UNSUPPORTED;
    }
    use_tc = true;
  } else if (path == ICD_PATH_AUTO) {
    use_tc = tensor_scan_supported(x->dim, k) && B > (have_master ? 2 : 4) && n >= 1024;
  }
  const bool scan_f32rows = !use_tc && have_master;
  const bool rescore_f32rows = have_master;
  // Where the tensor scan's scores are not the canonical products (fp32 master rows, or fp32 queries rounded to bf16)
  // its top-kc need not hold the exact top-k: finalise certifies each query and the exact stream scan re-searches the
  // others.  bf16 queries on bf16 rows score the canonical products themselves, and the k + 6 margin covers the fp32
  // accumulation order (DESIGN.md, "Exact search").
  const bool certify = use_tc && n > 0 && (have_master || !q_exact_bf16);

  // candidates per query kept by the scan
  int kc = k;
  if (use_tc) kc = std::min(ICD_MAX_K, (q_exact_bf16 && !have_master) ? k + 6 : 2 * k + 16);
  kc = std::max(kc, k);

  const int P = use_tc ? tensor_scan_max_partials() : stream_scan_grid();
  ICD_TRY(x->part_score.reserve((size_t)B * P * std::max(kc, use_tc ? tensor_scan_pre_slots() : kc) * 4));
  ICD_TRY(x->part_id.reserve((size_t)B * P * kc * 4));
  if (certify) {
    ICD_TRY(x->part_score.reserve((size_t)B * stream_scan_grid() * k * 4));
    ICD_TRY(x->part_id.reserve((size_t)B * stream_scan_grid() * k * 4));
  }
  ICD_TRY(x->cand_score.reserve((size_t)B * kc * 4));
  ICD_TRY(x->cand_id.reserve((size_t)B * kc * 8));

  if (x->timing) x->ev = x->ev_ring[x->timed_calls++ % icd_index::kTimingRing];
  cudaEvent_t* ev = x->ev;
  if (x->timing) cudaEventRecord(ev[0], st);
  const int64_t l0 = g_launches.load();

  int P_used = P;
  if (n == 0) {
    // nothing to scan: empty candidates
    ICD_CUDA(cudaMemsetAsync(x->cand_id.ptr, 0xff, (size_t)B * kc * 8, st));
    ICD_CUDA(cudaMemsetAsync(x->cand_score.ptr, 0, (size_t)B * kc * 4, st));
    if (x->timing) {
      cudaEventRecord(ev[1], st);
      cudaEventRecord(ev[2], st);
    }
  } else {
    if (use_tc) {
      if (!x->map_valid || x->map_gen != tensor_scan_generation()) {
        ICD_TRY(tensor_scan_make_map(x->tmap, x->table, n, x->dim));
        x->map_valid = true;
        x->map_gen = tensor_scan_generation();
        x->map_rows = n;
      }
      TensorScanArgs a{};
      a.table = x->table;
      a.levels = x->levels;
      a.n_rows = n;
      a.dim = x->dim;
      a.q_bf16 = x->q_bf16.ptr;
      a.B = B;
      a.k = kc;
      a.weight_pre = weight_pre;
      a.part_score = (float*)x->part_score.ptr;
      a.part_id = (int*)x->part_id.ptr;
      a.P = P;
      a.groups_used = &P_used;
      a.mask = d_mask;
      // [B] pruning bounds followed by the zeroed drift-limiter counters (two regions: pre-pass, main)
      const int prog_ints = tensor_scan_progress_ints();
      ICD_TRY(x->gbound.reserve(((size_t)B + 2 * prog_ints) * 4));
      ICD_CUDA(cudaMemsetAsync((int*)x->gbound.ptr + B, 0, (size_t)2 * prog_ints * 4, st));
      a.gbound = (int*)x->gbound.ptr;
      a.progress = (int*)x->gbound.ptr + B;
      const int sample = tensor_scan_sample_stride(n, kc);
      ICD_CUDA(cudaMemsetAsync(x->gbound.ptr, 0x80, (size_t)B * 4, st));
      if (sample > 1) {
        // sampling pre-pass over every `sample`-th row tile: a proven lower bound of the final kc-th best score per
        // query, so the main scan admits only rows that reach it (about kc * sample rows per query instead of every row
        // of each list's warm-up).  Slot maxima, no lists (scan_tc.cu, PRE; every kc <= 128); the list path (exact top-kc
        // of the sample, then the merge) remains behind icd_tune("scan_pre_slots", 0) for A/B.
        a.tile_stride = sample;
        if (kc <= tensor_scan_pre_capacity() && tensor_scan_pre_mode() != 0) {
          a.pre_slots = 1;
          ICD_TRY(launch_tensor_scan(a, x->tmap, st));
          a.pre_slots = 0;
          ICD_TRY(launch_bound_from_slots((const float*)x->part_score.ptr, B, P_used, tensor_scan_pre_slots(), kc,
                                          (int*)x->gbound.ptr, st));
        } else {
          ICD_TRY(launch_tensor_scan(a, x->tmap, st));
          MergeArgs m{};
          m.part_score = (const float*)x->part_score.ptr;
          m.part_id = (const int*)x->part_id.ptr;
          m.B = B;
          m.P = P_used;
          m.k_in = kc;
          m.k_out = kc;
          m.out_score = (float*)x->cand_score.ptr;
          m.out_id = (int64_t*)x->cand_id.ptr;
          m.row_offset = 0;
          m.bound_key_out = (int*)x->gbound.ptr;
          ICD_TRY(launch_merge(m, st));
        }
        a.tile_stride = 1;
        a.progress += prog_ints;
      }
      ICD_TRY(launch_tensor_scan(a, x->tmap, st));
    } else {
      const int per = stream_scan_max_queries(scan_f32rows, x->dim);
      for (int q0 = 0; q0 < B; q0 += per) {
        StreamScanArgs a{};
        a.table = scan_f32rows ? (const void*)x->master : (const void*)x->table;
        a.levels = x->levels;
        a.n_rows = n;
        a.dim = x->dim;
        a.f32rows = scan_f32rows;
        a.q = (const float*)x->q_f32.ptr + (size_t)q0 * x->dim;
        a.nq = std::min(per, B - q0);
        a.q0 = q0;
        a.k = kc;
        a.weight_pre = weight_pre;
        a.part_score = (float*)x->part_score.ptr;
        a.part_id = (int*)x->part_id.ptr;
        a.P = P;
        a.mask = d_mask;
        ICD_TRY(launch_stream_scan(a, st));
      }
    }
    if (x->timing) cudaEventRecord(ev[1], st);
    MergeArgs m{};
    m.part_score = (const float*)x->part_score.ptr;
    m.part_id = (const int*)x->part_id.ptr;
    m.B = B;
    m.P = P;  // unused tails of the P dimension are marked empty by the scan
    m.k_in = kc;
    m.k_out = kc;
    m.out_score = (float*)x->cand_score.ptr;
    m.out_id = (int64_t*)x->cand_id.ptr;
    m.row_offset = row_offset;
    if (use_tc && P_used < P) {
      // tensor scan wrote [B, P_used, kc] densely
      m.P = P_used;
    }
    ICD_TRY(launch_merge(m, st));
    if (x->timing) cudaEventRecord(ev[2], st);
  }

  FinaliseArgs f{};
  f.cand_score = (const float*)x->cand_score.ptr;
  f.cand_id = (const int64_t*)x->cand_id.ptr;
  f.cand_level = nullptr;
  f.S = 1;
  f.B = B;
  f.kcp = kc;
  f.k = k;
  f.row_offset = row_offset;
  f.n_local = n;
  f.q_f32 = (const float*)x->q_f32.ptr;
  f.rows = rescore_f32rows ? (const void*)x->master : (const void*)x->table;
  f.f32rows = rescore_f32rows;
  f.dim = x->dim;
  f.levels = x->levels;
  f.weight_mode = weight_mode;
  f.out_score = d_score;
  f.out_raw = d_raw;
  f.out_id = d_id;
  f.out_level = d_level;
  if (push) f.push = *push;
  if (certify) {
    ICD_CUDA(cudaMemsetAsync(x->fb.ptr, 0, 4, st));
    f.colstat = (const float*)x->colstat.ptr;
    f.fb = (int*)x->fb.ptr;
  }
  ICD_TRY(launch_finalise(f, st));
  if (certify) {
    // exact fallback for the uncertified queries, listed on the device: stream scan (one query per pass), merge and
    // finalise of list slot j into query fb[2 + j]'s result rows (and pushes, so a shard exchange sees only exact blocks)
    const int* fb = (const int*)x->fb.ptr;
    StreamScanArgs s{};
    s.table = have_master ? (const void*)x->master : (const void*)x->table;
    s.levels = x->levels;
    s.n_rows = n;
    s.dim = x->dim;
    s.f32rows = have_master;
    s.q = (const float*)x->q_f32.ptr;
    s.nq = B;
    s.k = k;
    s.weight_pre = weight_pre;
    s.part_score = (float*)x->part_score.ptr;
    s.part_id = (int*)x->part_id.ptr;
    s.P = stream_scan_grid();
    s.mask = d_mask;
    ICD_TRY(launch_stream_scan_listed(s, fb, st));
    MergeArgs m{};
    m.part_score = (const float*)x->part_score.ptr;
    m.part_id = (const int*)x->part_id.ptr;
    m.B = B;
    m.P = s.P;
    m.k_in = k;
    m.k_out = k;
    m.out_score = (float*)x->cand_score.ptr;
    m.out_id = (int64_t*)x->cand_id.ptr;
    m.row_offset = row_offset;
    m.count = fb;
    ICD_TRY(launch_merge(m, st));
    f.kcp = k;
    f.colstat = nullptr;
    f.fb = nullptr;
    f.fb_in = fb;
    ICD_TRY(launch_finalise(f, st));
  }
  if (x->timing) cudaEventRecord(ev[3], st);
  x->last_launches = (int)(g_launches.load() - l0);
  x->timing_pending = x->timing;
  return ICD_OK;
}

// stage queries (host or device, f32 or bf16) into the workspace as both fp32 and bf16
int index_stage_queries(icd_index* x, const void* q, int q_dtype, int B, cudaStream_t st) {
  const size_t ne = (size_t)B * x->dim;
  ICD_TRY(x->q_f32.reserve(ne * 4));
  ICD_TRY(x->q_bf16.reserve(ne * 2));
  const bool dev = is_device_ptr(q);
  if (q_dtype == ICD_F32) {
    if (dev) {
      ICD_CUDA(cudaMemcpyAsync(x->q_f32.ptr, q, ne * 4, cudaMemcpyDeviceToDevice, st));
    } else {
      ICD_CUDA(cudaMemcpyAsync(x->q_f32.ptr, q, ne * 4, cudaMemcpyHostToDevice, st));
    }
    ICD_TRY(launch_f32_to_bf16((const float*)x->q_f32.ptr, x->q_bf16.ptr, (int64_t)ne, st));
  } else if (q_dtype == ICD_BF16) {
    ICD_CUDA(cudaMemcpyAsync(x->q_bf16.ptr, q, ne * 2, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    ICD_TRY(launch_bf16_to_f32(x->q_bf16.ptr, (float*)x->q_f32.ptr, (int64_t)ne, st));
  } else {
    set_error("unknown query dtype %d", q_dtype);
    return ICD_E_ARG;
  }
  return ICD_OK;
}

int index_stage_mask(icd_index* x, const uint32_t* row_mask, int64_t mask_rows, const uint32_t** d_mask, cudaStream_t st) {
  *d_mask = nullptr;
  if (!row_mask) return ICD_OK;
  if (mask_rows != x->n) {
    set_error("row mask covers %lld rows, the table holds %lld", (long long)mask_rows, (long long)x->n);
    return ICD_E_ARG;
  }
  const size_t bytes = (size_t)((x->n + 31) / 32) * 4;
  if (is_device_ptr(row_mask)) {
    *d_mask = row_mask;
    return ICD_OK;
  }
  ICD_TRY(x->mask.reserve(std::max<size_t>(bytes, 16)));
  if (bytes) ICD_CUDA(cudaMemcpyAsync(x->mask.ptr, row_mask, bytes, cudaMemcpyHostToDevice, st));
  *d_mask = (const uint32_t*)x->mask.ptr;
  return ICD_OK;
}

int copy_out(void* dst, const void* src_dev, size_t bytes, cudaStream_t st) {
  if (!dst || dst == src_dev) return ICD_OK;
  ICD_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, is_device_ptr(dst) ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  return ICD_OK;
}

}  // namespace icd

using namespace icd;

extern "C" {

int icd_version(void) { return 100; }
const char* icd_last_error(void) { return t_error.c_str(); }
int64_t icd_launch_count(void) { return g_launches.load(); }
int icd_tune(const char* key, int value) {
  ICD_CHECK_ARG(key != nullptr, "key is null");
  if (!strcmp(key, "enc_pdl")) {
    encoder_set_pdl(value);
    return ICD_OK;
  }
  if (!strcmp(key, "enc_skinny")) {
    encoder_set_skinny(value);
    return ICD_OK;
  }
  if (tensor_scan_tune(key, value) != ICD_OK) {
    set_error("icd_tune: unknown key '%s'", key);
    return ICD_E_ARG;
  }
  return ICD_OK;
}
int icd_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int icd_index_create(int dim, int device, int64_t capacity_rows, int flags, icd_index** out) {
  ICD_CHECK_ARG(out != nullptr, "out is null");
  ICD_CHECK_ARG(dim >= 8 && dim % 8 == 0 && dim <= 1024, "dim must be a multiple of 8 in [8, 1024]");
  ICD_CHECK_ARG(capacity_rows >= 0 && capacity_rows <= 0x7fffffffLL, "capacity out of range");
  int ndev = 0;
  ICD_CUDA(cudaGetDeviceCount(&ndev));
  ICD_CHECK_ARG(device >= 0 && device < ndev, "no such CUDA device");
  DeviceGuard g(device);
  cudaDeviceProp prop;
  ICD_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("libicdrag is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    return ICD_E_UNSUPPORTED;
  }
  icd_index* x = new icd_index();
  x->dim = dim;
  x->device = device;
  x->flags = flags;
  int st = alloc_table(x, std::max<int64_t>(capacity_rows, 1024));
  if (st == ICD_OK) st = x->colstat.reserve((size_t)(2 * dim + 2) * 4);
  if (st == ICD_OK) st = x->fb.reserve((size_t)(2 + 8192) * 4);
  if (st == ICD_OK && (cudaMemset(x->colstat.ptr, 0, (size_t)(2 * dim + 2) * 4) != cudaSuccess ||
                       cudaMemset(x->fb.ptr, 0, 8) != cudaSuccess)) {
    set_error("icd_index_create: cudaMemset failed");
    st = ICD_E_CUDA;
  }
  if (st != ICD_OK) {
    if (x->table) cudaFree(x->table);
    if (x->master) cudaFree(x->master);
    if (x->levels) cudaFree(x->levels);
    x->colstat.release();
    x->fb.release();
    delete x;
    return st;
  }
  for (int r = 0; r < icd_index::kTimingRing; ++r)
    for (int i = 0; i < 4; ++i) cudaEventCreate(&x->ev_ring[r][i]);
  *out = x;
  return ICD_OK;
}

int icd_index_destroy(icd_index* x) {
  if (!x) return ICD_OK;
  DeviceGuard g(x->device);
  cudaDeviceSynchronize();
  if (!x->adopted) {
    if (x->table) cudaFree(x->table);
    if (x->levels) cudaFree(x->levels);
  }
  if (x->master) cudaFree(x->master);
  x->q_f32.release();
  x->q_bf16.release();
  x->part_score.release();
  x->part_id.release();
  x->cand_score.release();
  x->cand_id.release();
  x->out_stage.release();
  x->in_stage.release();
  x->gbound.release();
  x->mask.release();
  x->colstat.release();
  x->fb.release();
  x->q_f32_alt.release();
  x->q_bf16_alt.release();
  x->out_stage_alt.release();
  x->page_ws.release();
  if (x->copy_stream) cudaStreamDestroy(x->copy_stream);
  for (int i = 0; i < 2; ++i) {
    if (x->ev_ready[i]) cudaEventDestroy(x->ev_ready[i]);
    if (x->ev_done[i]) cudaEventDestroy(x->ev_done[i]);
  }
  for (int r = 0; r < icd_index::kTimingRing; ++r)
    for (int i = 0; i < 4; ++i) cudaEventDestroy(x->ev_ring[r][i]);
  delete x;
  return ICD_OK;
}

int icd_index_append(icd_index* x, const void* vecs, int dtype, const uint8_t* level, int64_t n) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  ICD_CHECK_ARG(n >= 0, "negative row count");
  if (n == 0) return ICD_OK;
  ICD_CHECK_ARG(vecs != nullptr, "vecs is null");
  ICD_CHECK_ARG(dtype == ICD_F32 || dtype == ICD_BF16, "unknown dtype");
  if (x->adopted) {
    set_error("append on an adopted table");
    return ICD_E_STATE;
  }
  ICD_CHECK_ARG(x->n + n <= 0x7fffffffLL, "table would exceed 2^31 rows");
  DeviceGuard g(x->device);
  if (x->n + n > x->cap) ICD_TRY(alloc_table(x, std::max<int64_t>(x->cap * 2, x->n + n)));
  const size_t ne = (size_t)n * x->dim;
  const bool dev = is_device_ptr(vecs);
  char* t_dst = (char*)x->table + (size_t)x->n * x->dim * 2;
  cudaStream_t st = 0;
  if (dtype == ICD_BF16) {
    ICD_CUDA(cudaMemcpyAsync(t_dst, vecs, ne * 2, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    if (x->master) ICD_TRY(launch_bf16_to_f32(t_dst, x->master + (size_t)x->n * x->dim, (int64_t)ne, st));
  } else {
    const float* src = (const float*)vecs;
    if (x->master) {
      float* m_dst = x->master + (size_t)x->n * x->dim;
      ICD_CUDA(cudaMemcpyAsync(m_dst, vecs, ne * 4, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
      src = m_dst;
    } else if (!dev) {
      ICD_TRY(x->in_stage.reserve(ne * 4));
      ICD_CUDA(cudaMemcpyAsync(x->in_stage.ptr, vecs, ne * 4, cudaMemcpyHostToDevice, st));
      src = (const float*)x->in_stage.ptr;
    }
    ICD_TRY(launch_f32_to_bf16(src, t_dst, (int64_t)ne, st));
  }
  if (level) {
    ICD_CUDA(cudaMemcpyAsync(x->levels + x->n, level, n, is_device_ptr(level) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
  } else {
    ICD_CUDA(cudaMemsetAsync(x->levels + x->n, 1, n, st));
  }
  ICD_TRY(launch_column_stats(x->table, x->master, x->n, n, x->dim, (float*)x->colstat.ptr, st));
  ICD_CUDA(cudaStreamSynchronize(st));
  x->n += n;
  x->map_valid = false;
  return ICD_OK;
}

int icd_index_adopt(icd_index* x, const void* dev_bf16, const uint8_t* dev_level, int64_t n) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  ICD_CHECK_ARG(n >= 0 && n <= 0x7fffffffLL, "row count out of range");
  ICD_CHECK_ARG(dev_bf16 != nullptr && dev_level != nullptr, "null table");
  ICD_CHECK_ARG(is_device_ptr(dev_bf16) && is_device_ptr(dev_level), "adopt needs device pointers");
  ICD_CHECK_ARG(((uintptr_t)dev_bf16 & 127) == 0, "table must be 128-byte aligned");
  if (x->flags & ICD_INDEX_KEEP_F32) {
    set_error("adopt is not available with ICD_INDEX_KEEP_F32");
    return ICD_E_STATE;
  }
  DeviceGuard g(x->device);
  if (!x->adopted) {
    if (x->table) cudaFree(x->table);
    if (x->levels) cudaFree(x->levels);
  }
  x->table = const_cast<void*>(dev_bf16);
  x->levels = const_cast<uint8_t*>(dev_level);
  x->adopted = true;
  x->n = n;
  x->cap = n;
  x->map_valid = false;
  ICD_CUDA(cudaMemset(x->colstat.ptr, 0, (size_t)(2 * x->dim + 2) * 4));
  ICD_TRY(launch_column_stats(x->table, nullptr, 0, n, x->dim, (float*)x->colstat.ptr, 0));
  ICD_CUDA(cudaStreamSynchronize(0));
  return ICD_OK;
}

int icd_index_clear(icd_index* x) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  if (x->adopted) {
    set_error("clear on an adopted table");
    return ICD_E_STATE;
  }
  x->n = 0;
  x->map_valid = false;
  DeviceGuard g(x->device);
  ICD_CUDA(cudaMemset(x->colstat.ptr, 0, (size_t)(2 * x->dim + 2) * 4));
  return ICD_OK;
}

int icd_index_take_fallbacks(icd_index* x, int64_t* count) {
  ICD_CHECK_ARG(x != nullptr && count != nullptr, "null argument");
  DeviceGuard g(x->device);
  int v = 0;
  ICD_CUDA(cudaDeviceSynchronize());
  ICD_CUDA(cudaMemcpy(&v, (const int*)x->fb.ptr + 1, 4, cudaMemcpyDeviceToHost));
  ICD_CUDA(cudaMemset((int*)x->fb.ptr + 1, 0, 4));
  *count = v;
  return ICD_OK;
}

int64_t icd_index_size(const icd_index* x) { return x ? x->n : -1; }
int icd_index_dim(const icd_index* x) { return x ? x->dim : -1; }

int icd_index_read(const icd_index* x, int64_t row0, int64_t n, float* out) {
  ICD_CHECK_ARG(x != nullptr && out != nullptr, "null argument");
  ICD_CHECK_ARG(row0 >= 0 && n >= 0 && row0 + n <= x->n, "row range out of bounds");
  if (n == 0) return ICD_OK;
  DeviceGuard g(x->device);
  const size_t ne = (size_t)n * x->dim;
  const bool dev = is_device_ptr(out);
  if (x->master) {
    ICD_CUDA(cudaMemcpy(out, x->master + (size_t)row0 * x->dim, ne * 4, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost));
    return ICD_OK;
  }
  float* tmp = out;
  if (!dev) ICD_CUDA(cudaMalloc((void**)&tmp, ne * 4));
  int st = launch_bf16_to_f32((const char*)x->table + (size_t)row0 * x->dim * 2, tmp, (int64_t)ne, 0);
  if (st == ICD_OK && !dev) {
    cudaError_t e = cudaMemcpy(out, tmp, ne * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      set_error("icd_index_read: %s", cudaGetErrorString(e));
      st = ICD_E_CUDA;
    }
  } else if (st == ICD_OK) {
    cudaDeviceSynchronize();
  }
  if (!dev) cudaFree(tmp);
  return st;
}

namespace icd {

// Large batch, queries AND results in host memory (MilvusService.search_batch with numpy arrays: BASELINE configs[1] moves
// 30 MB of fp32 queries): chunks of kPipeChunk queries on two streams, so that the host-to-device copy of chunk c + 1 runs
// under the scan of chunk c.  Two sets of staging buffers alternate; the device-to-host copy of chunk c goes to the copy
// stream after chunk c + 1 has been enqueued (with pageable destinations it blocks the calling thread until chunk c is
// done; issued earlier it would hold back the next chunk's copy-in).  r02x measured 4.45 ms per 10 000 queries against
// 1.53 ms with resident buffers before this.
constexpr int kPipeChunk = 2048;

static int search_host_pipelined(icd_index* x, const void* q, int q_dtype, int B, int k, int weight_mode, int path,
                                 const uint32_t* d_mask, float* out_score, float* out_raw, int64_t* out_id, cudaStream_t st) {
  if (!x->copy_stream) {
    ICD_CUDA(cudaStreamCreateWithFlags(&x->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      ICD_CUDA(cudaEventCreateWithFlags(&x->ev_ready[i], cudaEventDisableTiming));
      ICD_CUDA(cudaEventCreateWithFlags(&x->ev_done[i], cudaEventDisableTiming));
    }
  }
  const size_t esz = q_dtype == ICD_F32 ? 4 : 2;
  const size_t qbytes = (size_t)kPipeChunk * x->dim;
  ICD_TRY(x->q_f32.reserve(qbytes * 4));
  ICD_TRY(x->q_bf16.reserve(qbytes * 2));
  ICD_TRY(x->q_f32_alt.reserve(qbytes * 4));
  ICD_TRY(x->q_bf16_alt.reserve(qbytes * 2));
  ICD_TRY(x->out_stage.reserve((size_t)kPipeChunk * k * 16));
  ICD_TRY(x->out_stage_alt.reserve((size_t)kPipeChunk * k * 16));
  auto swap_sets = [&]() {
    std::swap(x->q_f32, x->q_f32_alt);
    std::swap(x->q_bf16, x->q_bf16_alt);
    std::swap(x->out_stage, x->out_stage_alt);
  };
  // everything already enqueued on st (it may still be reading the staging buffers) comes first
  ICD_CUDA(cudaEventRecord(x->ev_done[0], st));
  ICD_CUDA(cudaStreamWaitEvent(x->copy_stream, x->ev_done[0], 0));
  struct Pending {
    int b0 = 0, nb = 0, set = 0;
    float* d_score = nullptr;
  } prev;
  // results of a finished chunk -> host, on the COPY stream behind the event recorded after that chunk's search: a copy
  // into pageable memory blocks the calling thread until it is done, and on st it would sit behind the NEXT chunk's scan
  auto copy_back = [&](const Pending& c) -> int {
    if (c.nb == 0) return ICD_OK;
    const float* d_raw = c.d_score + (size_t)c.nb * k;
    const int64_t* d_id = reinterpret_cast<const int64_t*>(d_raw + (size_t)c.nb * k);
    cudaStream_t cs = x->copy_stream;
    ICD_CUDA(cudaStreamWaitEvent(cs, x->ev_done[c.set], 0));
    if (out_score) ICD_CUDA(cudaMemcpyAsync(out_score + (size_t)c.b0 * k, c.d_score, (size_t)c.nb * k * 4, cudaMemcpyDeviceToHost, cs));
    if (out_raw) ICD_CUDA(cudaMemcpyAsync(out_raw + (size_t)c.b0 * k, d_raw, (size_t)c.nb * k * 4, cudaMemcpyDeviceToHost, cs));
    if (out_id) ICD_CUDA(cudaMemcpyAsync(out_id + (size_t)c.b0 * k, d_id, (size_t)c.nb * k * 8, cudaMemcpyDeviceToHost, cs));
    return ICD_OK;
  };
  int status = ICD_OK, chunk = 0;
  for (int b0 = 0; b0 < B && status == ICD_OK; b0 += kPipeChunk, ++chunk) {
    const int nb = std::min(kPipeChunk, B - b0);
    const int s = chunk & 1;
    if (s) swap_sets();   // this chunk works in the alternate set
    const size_t ne = (size_t)nb * x->dim;
    void* d_in = q_dtype == ICD_F32 ? x->q_f32.ptr : x->q_bf16.ptr;
    auto body = [&]() -> int {
      // copy stream: [copy-in c] [copy-back c - 1] [copy-in c + 1] ... -- the copy-in of chunk c + 2 into this set is
      // therefore behind the copy-back of chunk c, which is behind chunk c's search
      ICD_CUDA(cudaMemcpyAsync(d_in, (const char*)q + (size_t)b0 * x->dim * esz, ne * esz, cudaMemcpyHostToDevice, x->copy_stream));
      ICD_CUDA(cudaEventRecord(x->ev_ready[s], x->copy_stream));
      ICD_CUDA(cudaStreamWaitEvent(st, x->ev_ready[s], 0));
      if (q_dtype == ICD_F32) ICD_TRY(launch_f32_to_bf16((const float*)x->q_f32.ptr, x->q_bf16.ptr, (int64_t)ne, st));
      else ICD_TRY(launch_bf16_to_f32(x->q_bf16.ptr, (float*)x->q_f32.ptr, (int64_t)ne, st));
      float* d_score = (float*)x->out_stage.ptr;
      float* d_raw = d_score + (size_t)nb * k;
      int64_t* d_id = (int64_t*)(d_raw + (size_t)nb * k);
      ICD_TRY(index_search_device(x, nb, k, weight_mode, path, 0, d_score, d_raw, d_id, nullptr, q_dtype == ICD_BF16, nullptr,
                                  d_mask, st));
      ICD_CUDA(cudaEventRecord(x->ev_done[s], st));
      ICD_TRY(copy_back(prev));   // the previous chunk's results, while this chunk is being searched
      prev.b0 = b0, prev.nb = nb, prev.set = s, prev.d_score = d_score;
      return ICD_OK;
    };
    status = body();
    if (s) swap_sets();
  }
  if (status == ICD_OK) status = copy_back(prev);
  cudaError_t e = cudaStreamSynchronize(st);   // also on failure: nothing may still be using the staging sets
  cudaStreamSynchronize(x->copy_stream);
  if (status == ICD_OK && e != cudaSuccess) {
    set_error("icd_index_search: %s", cudaGetErrorString(e));
    status = ICD_E_CUDA;
  }
  return status;
}

}  // namespace icd

int icd_index_search(icd_index* x, const void* q, int q_dtype, int B, int k, int weight_mode, int path,
                     float* out_score, float* out_raw, int64_t* out_id, void* stream, int sync) {
  return icd_index_search_filtered(x, q, q_dtype, B, k, weight_mode, path, nullptr, 0, out_score, out_raw, out_id, stream,
                                   sync);
}

int icd_index_search_filtered(icd_index* x, const void* q, int q_dtype, int B, int k, int weight_mode, int path,
                              const uint32_t* row_mask, int64_t mask_rows, float* out_score, float* out_raw,
                              int64_t* out_id, void* stream, int sync) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  ICD_CHECK_ARG(B >= 0, "negative batch");
  ICD_CHECK_ARG(k >= 1 && k <= ICD_MAX_K, "k must be in [1, 128]");
  ICD_CHECK_ARG(weight_mode >= 0 && weight_mode <= 2, "unknown weight mode");
  ICD_CHECK_ARG(path >= 0 && path <= 2, "unknown path");
  if (B == 0) return ICD_OK;
  ICD_CHECK_ARG(q != nullptr, "q is null");
  DeviceGuard g(x->device);
  cudaStream_t st = (cudaStream_t)stream;
  const bool host_out = (out_score && !is_device_ptr(out_score)) || (out_raw && !is_device_ptr(out_raw)) ||
                        (out_id && !is_device_ptr(out_id));
  const bool all_host_out = (!out_score || !is_device_ptr(out_score)) && (!out_raw || !is_device_ptr(out_raw)) &&
                            (!out_id || !is_device_ptr(out_id));
  const uint32_t* d_mask = nullptr;
  ICD_TRY(index_stage_mask(x, row_mask, mask_rows, &d_mask, st));
  if (B >= 2 * kPipeChunk && !is_device_ptr(q) && all_host_out && x->n > 0)
    return search_host_pipelined(x, q, q_dtype, B, k, weight_mode, path, d_mask, out_score, out_raw, out_id, st);
  constexpr int kMaxBatch = 8192;  // bounds the workspace; larger batches run as several passes
  for (int b0 = 0; b0 < B; b0 += kMaxBatch) {
    const int nb = std::min(kMaxBatch, B - b0);
    const size_t qoff = (size_t)b0 * x->dim * (q_dtype == ICD_F32 ? 4 : 2);
    ICD_TRY(index_stage_queries(x, (const char*)q + qoff, q_dtype, nb, st));
    // device-side result buffers: caller's when on device, staging otherwise
    ICD_TRY(x->out_stage.reserve((size_t)nb * k * 16));
    float* d_score = (float*)x->out_stage.ptr;
    float* d_raw = d_score + (size_t)nb * k;
    int64_t* d_id = (int64_t*)(d_raw + (size_t)nb * k);
    float* o_score = out_score ? out_score + (size_t)b0 * k : nullptr;
    float* o_raw = out_raw ? out_raw + (size_t)b0 * k : nullptr;
    int64_t* o_id = out_id ? out_id + (size_t)b0 * k : nullptr;
    float* k_score = (o_score && is_device_ptr(o_score)) ? o_score : (o_score ? d_score : nullptr);
    float* k_raw = (o_raw && is_device_ptr(o_raw)) ? o_raw : (o_raw ? d_raw : nullptr);
    int64_t* k_id = (o_id && is_device_ptr(o_id)) ? o_id : (o_id ? d_id : nullptr);
    ICD_TRY(index_search_device(x, nb, k, weight_mode, path, 0, k_score, k_raw, k_id, nullptr,
                                q_dtype == ICD_BF16, nullptr, d_mask, st));
    ICD_TRY(copy_out(o_score, k_score, (size_t)nb * k * 4, st));
    ICD_TRY(copy_out(o_raw, k_raw, (size_t)nb * k * 4, st));
    ICD_TRY(copy_out(o_id, k_id, (size_t)nb * k * 8, st));
    if (B > kMaxBatch) ICD_CUDA(cudaStreamSynchronize(st));  // staging buffers are reused
  }
  if (sync || host_out || !is_device_ptr(q)) ICD_CUDA(cudaStreamSynchronize(st));
  return ICD_OK;
}

int icd_index_search_page(icd_index* x, const void* q, int q_dtype, int B, const icd_search_page* page, int weight_mode,
                          const uint32_t* row_mask, int64_t mask_rows, float* out_score, float* out_raw, int64_t* out_id,
                          void* stream, int sync) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  ICD_CHECK_ARG(page != nullptr, "page is null");
  ICD_CHECK_ARG(B >= 0, "negative batch");
  ICD_CHECK_ARG(page->limit >= 1, "limit must be >= 1");
  ICD_CHECK_ARG(page->offset >= 0, "offset must be >= 0");
  ICD_CHECK_ARG((int64_t)page->offset + page->limit <= ICD_MAX_LIMIT, "offset + limit must be <= 16384");
  ICD_CHECK_ARG((page->range_flags & ~(ICD_RANGE_RADIUS | ICD_RANGE_FILTER)) == 0, "unknown range flags");
  ICD_CHECK_ARG(page->range_flags != (ICD_RANGE_RADIUS | ICD_RANGE_FILTER) || page->radius < page->range_filter,
                "radius must be below range_filter");
  ICD_CHECK_ARG(weight_mode >= 0 && weight_mode <= 2, "unknown weight mode");
  if (row_mask && mask_rows != x->n) {
    set_error("row mask covers %lld rows, the table holds %lld", (long long)mask_rows, (long long)x->n);
    return ICD_E_ARG;
  }
  if (B == 0) return ICD_OK;
  ICD_CHECK_ARG(q != nullptr, "q is null");
  DeviceGuard g(x->device);
  cudaStream_t st = (cudaStream_t)stream;
  const int limit = page->limit, K = page->offset + page->limit;
  const bool host_out = (out_score && !is_device_ptr(out_score)) || (out_raw && !is_device_ptr(out_raw)) ||
                        (out_id && !is_device_ptr(out_id));
  const uint32_t* d_mask = nullptr;
  ICD_TRY(index_stage_mask(x, row_mask, mask_rows, &d_mask, st));
  constexpr int kMaxBatch = 8192;  // bounds the query staging; larger batches run as several passes
  const int chunk = page_search_chunk(x->n, K, std::min(B, kMaxBatch));
  const size_t ws_bytes = page_search_workspace_bytes(x->n, K, chunk);
  ICD_TRY(x->page_ws.reserve(ws_bytes));
  for (int b0 = 0; b0 < B; b0 += kMaxBatch) {
    const int nb = std::min(kMaxBatch, B - b0);
    const size_t qoff = (size_t)b0 * x->dim * (q_dtype == ICD_F32 ? 4 : 2);
    ICD_TRY(index_stage_queries(x, (const char*)q + qoff, q_dtype, nb, st));
    // device-side result buffers: caller's when on device, staging otherwise
    ICD_TRY(x->out_stage.reserve((size_t)nb * limit * 16));
    float* d_score = (float*)x->out_stage.ptr;
    float* d_raw = d_score + (size_t)nb * limit;
    int64_t* d_id = (int64_t*)(d_raw + (size_t)nb * limit);
    float* o_score = out_score ? out_score + (size_t)b0 * limit : nullptr;
    float* o_raw = out_raw ? out_raw + (size_t)b0 * limit : nullptr;
    int64_t* o_id = out_id ? out_id + (size_t)b0 * limit : nullptr;
    PageSearchArgs a{};
    a.rows = x->master ? (const void*)x->master : (const void*)x->table;
    a.f32rows = x->master != nullptr;
    a.levels = x->levels;
    a.n = x->n;
    a.dim = x->dim;
    a.q = (const float*)x->q_f32.ptr;
    a.nq = nb;
    a.mask = d_mask;
    a.range_flags = page->range_flags;
    a.radius = page->radius;
    a.range_filter = page->range_filter;
    a.weight_mode = weight_mode;
    a.offset = page->offset;
    a.limit = limit;
    a.chunk = chunk;
    a.workspace = x->page_ws.ptr;
    a.workspace_bytes = x->page_ws.cap;
    a.out_score = (o_score && is_device_ptr(o_score)) ? o_score : (o_score ? d_score : nullptr);
    a.out_raw = (o_raw && is_device_ptr(o_raw)) ? o_raw : (o_raw ? d_raw : nullptr);
    a.out_id = (o_id && is_device_ptr(o_id)) ? o_id : (o_id ? d_id : nullptr);
    ICD_TRY(launch_page_search(a, st));
    ICD_TRY(copy_out(o_score, a.out_score, (size_t)nb * limit * 4, st));
    ICD_TRY(copy_out(o_raw, a.out_raw, (size_t)nb * limit * 4, st));
    ICD_TRY(copy_out(o_id, a.out_id, (size_t)nb * limit * 8, st));
    if (B > kMaxBatch) ICD_CUDA(cudaStreamSynchronize(st));  // staging buffers are reused
  }
  if (sync || host_out || !is_device_ptr(q)) ICD_CUDA(cudaStreamSynchronize(st));
  return ICD_OK;
}

int icd_index_set_timing(icd_index* x, int enabled) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  x->timing = enabled != 0;
  x->timed_calls = 0;
  x->timing_pending = false;
  return ICD_OK;
}

int icd_index_mean_timing(const icd_index* x, float* us3, int* calls) {
  ICD_CHECK_ARG(x != nullptr && us3 != nullptr, "null argument");
  us3[0] = us3[1] = us3[2] = 0.f;
  const int n = (int)std::min<int64_t>(x->timed_calls, icd_index::kTimingRing);
  if (calls) *calls = n;
  if (n == 0 || !x->timing_pending) return ICD_OK;
  DeviceGuard g(x->device);
  ICD_CUDA(cudaEventSynchronize(x->ev[3]));
  double acc[3] = {0, 0, 0};
  for (int c = 0; c < n; ++c) {
    const cudaEvent_t* q = x->ev_ring[(x->timed_calls - 1 - c) % icd_index::kTimingRing];
    for (int i = 0; i < 3; ++i) {
      float ms = 0.f;
      ICD_CUDA(cudaEventElapsedTime(&ms, q[i], q[i + 1]));
      acc[i] += ms;
    }
  }
  for (int i = 0; i < 3; ++i) us3[i] = (float)(acc[i] * 1000.0 / n);
  return ICD_OK;
}

int icd_index_last_timing(const icd_index* x, float* us3, int* launches) {
  ICD_CHECK_ARG(x != nullptr, "index is null");
  if (launches) *launches = x->last_launches;
  if (us3) {
    us3[0] = us3[1] = us3[2] = 0.f;
    if (x->timing_pending) {
      DeviceGuard g(x->device);
      ICD_CUDA(cudaEventSynchronize(x->ev[3]));
      for (int i = 0; i < 3; ++i) {
        float ms = 0.f;
        ICD_CUDA(cudaEventElapsedTime(&ms, x->ev[i], x->ev[i + 1]));
        us3[i] = ms * 1000.f;
      }
    }
  }
  return ICD_OK;
}

}  // extern "C"
