// api_shard.cu -- row-sharded scan over the GPUs of one box (include/icdrag.h, icd_shard_group_*).
//
// New work: the reference is single-process (SURVEY.md section 5).  Rank r scans its own rows
// with the local kernels, keeps k exact-rescored candidates per query, exchanges them and
// merges.  Two exchanges:
//   0  three grouped ncclAllGather calls (raw f32, id i64, level u8) + merge kernel
//   1  fused: the local finalise kernel stores each query's block straight into every peer's
//      receive slab through cudaIpc-mapped pointers over NVLink and releases a per-query flag;
//      the merge kernel acquires the flags of the sources it needs -- no collective call, no
//      host synchronisation, query-granular overlap.
// NCCL is resolved at run time (dlopen) so the library has no link-time dependency on it.
#include <dlfcn.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "index_impl.h"
#include "kernels.h"

namespace icd {

struct NcclId {
  char internal[ICD_NCCL_ID_BYTES];
};
typedef void* ncclComm_t;
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, NcclId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl() {
  if (g_nccl.handle) return ICD_OK;
  const char* env = getenv("ICDRAG_NCCL_LIB");
  const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n || !*n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) {
    set_error("cannot dlopen NCCL (set ICDRAG_NCCL_LIB): %s", dlerror());
    return ICD_E_NCCL;
  }
  NcclApi a;
  a.handle = h;
  a.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
  a.CommInitRank = (int (*)(ncclComm_t*, int, NcclId, int))dlsym(h, "ncclCommInitRank");
  a.CommDestroy = (int (*)(ncclComm_t))dlsym(h, "ncclCommDestroy");
  a.AllGather = (int (*)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t))dlsym(h, "ncclAllGather");
  a.GroupStart = (int (*)())dlsym(h, "ncclGroupStart");
  a.GroupEnd = (int (*)())dlsym(h, "ncclGroupEnd");
  a.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllGather || !a.GroupStart || !a.GroupEnd) {
    set_error("NCCL library lacks required symbols");
    return ICD_E_NCCL;
  }
  g_nccl = a;
  return ICD_OK;
}

#define ICD_NCCL(expr)                                                                          \
  do {                                                                                          \
    int _r = (expr);                                                                            \
    if (_r != 0) {                                                                              \
      icd::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                              \
                     icd::g_nccl.GetErrorString ? icd::g_nccl.GetErrorString(_r) : "nccl error"); \
      return ICD_E_NCCL;                                                                        \
    }                                                                                           \
  } while (0)

constexpr int kSlabMaxB = 8192;  // queries per pass
constexpr int kMaxWorld = 8;

// receive slab of one rank: [parity 2][source world] blocks of (raw, id, level) + flags
struct SlabLayout {
  int world;
  size_t blk_raw, blk_id, blk_lv, blk_flag, blk_total, total;
  explicit SlabLayout(int w) : world(w) {
    const size_t n = (size_t)kSlabMaxB * ICD_MAX_K;
    blk_raw = 0;
    blk_id = blk_raw + n * 4;
    blk_lv = blk_id + n * 8;
    blk_flag = (blk_lv + n + 255) & ~(size_t)255;
    blk_total = (blk_flag + (size_t)kSlabMaxB * 4 + 255) & ~(size_t)255;
    total = blk_total * 2 * w;
  }
  size_t block(int parity, int src) const { return ((size_t)parity * world + src) * blk_total; }
};

}  // namespace icd

struct icd_shard_group {
  int rank = 0, world = 1;
  int64_t row_offset = 0;
  icd_index* local = nullptr;
  icd::ncclComm_t comm = nullptr;
  // exchange buffers (NCCL path): send [B,k] triple, recv [world][B,k] triple
  icd::DeviceBuf send_raw, send_id, send_lv, recv_raw, recv_id, recv_lv, out_stage;
  // peer path
  char* slab = nullptr;
  char* peer_slab[icd::kMaxWorld] = {nullptr};
  bool peers_open = false;
  uint32_t epoch = 0;
};

using namespace icd;

extern "C" {

int icd_nccl_unique_id(void* out128) {
  ICD_CHECK_ARG(out128 != nullptr, "null argument");
  ICD_TRY(load_nccl());
  NcclId id;
  ICD_NCCL(g_nccl.GetUniqueId(&id));
  memcpy(out128, &id, sizeof(id));
  return ICD_OK;
}

int icd_shard_group_create(const void* nccl_id128, int rank, int world, int64_t row_offset, icd_index* local,
                           icd_shard_group** out) {
  ICD_CHECK_ARG(out && local, "null argument");
  ICD_CHECK_ARG(world >= 1 && world <= kMaxWorld && rank >= 0 && rank < world, "bad rank/world");
  ICD_CUDA(cudaSetDevice(local->device));
  icd_shard_group* g = new icd_shard_group();
  g->rank = rank;
  g->world = world;
  g->row_offset = row_offset;
  g->local = local;
  if (nccl_id128) {
    int st = load_nccl();
    if (st != ICD_OK) {
      delete g;
      return st;
    }
    NcclId id;
    memcpy(&id, nccl_id128, sizeof(id));
    int r = g_nccl.CommInitRank(&g->comm, world, id, rank);
    if (r != 0) {
      set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?");
      delete g;
      return ICD_E_NCCL;
    }
  }
  *out = g;
  return ICD_OK;
}

int icd_shard_group_destroy(icd_shard_group* g) {
  if (!g) return ICD_OK;
  cudaSetDevice(g->local->device);
  cudaDeviceSynchronize();
  if (g->peers_open) {
    for (int r = 0; r < g->world; ++r)
      if (r != g->rank && g->peer_slab[r]) cudaIpcCloseMemHandle(g->peer_slab[r]);
  }
  if (g->slab) cudaFree(g->slab);
  if (g->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(g->comm);
  g->send_raw.release();
  g->send_id.release();
  g->send_lv.release();
  g->recv_raw.release();
  g->recv_id.release();
  g->recv_lv.release();
  g->out_stage.release();
  delete g;
  return ICD_OK;
}

int icd_shard_group_export_slab(icd_shard_group* g, void* out_handle64) {
  ICD_CHECK_ARG(g && out_handle64, "null argument");
  ICD_CUDA(cudaSetDevice(g->local->device));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  if (!g->slab) {
    SlabLayout L(g->world);
    ICD_CUDA(cudaMalloc((void**)&g->slab, L.total));
    ICD_CUDA(cudaMemset(g->slab, 0, L.total));
  }
  cudaIpcMemHandle_t h;
  ICD_CUDA(cudaIpcGetMemHandle(&h, g->slab));
  memcpy(out_handle64, &h, 64);
  return ICD_OK;
}

int icd_shard_group_import_slabs(icd_shard_group* g, const void* handles) {
  ICD_CHECK_ARG(g && handles, "null argument");
  if (!g->slab) {
    set_error("export the local slab before importing the peers'");
    return ICD_E_STATE;
  }
  ICD_CUDA(cudaSetDevice(g->local->device));
  for (int r = 0; r < g->world; ++r) {
    if (r == g->rank) {
      g->peer_slab[r] = g->slab;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, (const char*)handles + (size_t)r * 64, 64);
    void* p = nullptr;
    ICD_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    g->peer_slab[r] = (char*)p;
  }
  g->peers_open = true;
  return ICD_OK;
}

int icd_shard_group_search(icd_shard_group* g, const void* q, int q_dtype, int B, int k, int weight_mode, int path,
                           int exchange, float* out_score, float* out_raw, int64_t* out_id, void* stream, int sync) {
  return icd_shard_group_search_filtered(g, q, q_dtype, B, k, weight_mode, path, exchange, nullptr, 0, out_score, out_raw,
                                         out_id, stream, sync);
}

int icd_shard_group_search_filtered(icd_shard_group* g, const void* q, int q_dtype, int B, int k, int weight_mode,
                                    int path, int exchange, const uint32_t* row_mask, int64_t mask_rows,
                                    float* out_score, float* out_raw, int64_t* out_id, void* stream, int sync) {
  ICD_CHECK_ARG(g != nullptr, "group is null");
  ICD_CHECK_ARG(B >= 0 && B <= kSlabMaxB, "batch must be in [0, 8192] per call");
  ICD_CHECK_ARG(k >= 1 && k <= ICD_MAX_K, "k must be in [1, 128]");
  ICD_CHECK_ARG(weight_mode >= 0 && weight_mode <= 2, "unknown weight mode");
  ICD_CHECK_ARG(exchange == 0 || exchange == 1, "unknown exchange");
  if (B == 0) return ICD_OK;
  ICD_CHECK_ARG(q != nullptr, "q is null");
  icd_index* x = g->local;
  ICD_CUDA(cudaSetDevice(x->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int W = g->world;
  if (exchange == 0 && W > 1 && !g->comm) {
    set_error("group was created without an NCCL id");
    return ICD_E_STATE;
  }
  if (exchange == 1 && W > 1 && !g->peers_open) {
    set_error("peer slabs not imported");
    return ICD_E_STATE;
  }
  ICD_TRY(index_stage_queries(x, q, q_dtype, B, st));
  const uint32_t* d_mask = nullptr;   // this rank's local rows
  ICD_TRY(index_stage_mask(x, row_mask, mask_rows, &d_mask, st));
  const size_t nk = (size_t)B * k;
  const int local_mode = (weight_mode == ICD_WEIGHT_PRE) ? ICD_WEIGHT_PRE : ICD_WEIGHT_NONE;

  // device-side outputs
  ICD_TRY(g->out_stage.reserve(nk * 16));
  float* d_score = (float*)g->out_stage.ptr;
  float* d_raw = d_score + nk;
  int64_t* d_id = (int64_t*)(d_raw + nk);
  float* k_score = (out_score && is_device_ptr(out_score)) ? out_score : d_score;
  float* k_raw = (out_raw && is_device_ptr(out_raw)) ? out_raw : d_raw;
  int64_t* k_id = (out_id && is_device_ptr(out_id)) ? out_id : d_id;

  FinaliseArgs f{};
  f.S = W;
  f.B = B;
  f.kcp = k;
  f.k = k;
  f.row_offset = g->row_offset;
  f.n_local = x->n;
  f.q_f32 = nullptr;  // candidates arrive exactly rescored by their owners
  f.rows = nullptr;
  f.dim = x->dim;
  f.levels = nullptr;
  f.weight_mode = weight_mode;
  f.out_score = k_score;
  f.out_raw = k_raw;
  f.out_id = k_id;
  f.out_level = nullptr;

  if (exchange == 0 || W == 1) {
    ICD_TRY(g->send_raw.reserve(nk * 4));
    ICD_TRY(g->send_id.reserve(nk * 8));
    ICD_TRY(g->send_lv.reserve(nk));
    ICD_TRY(g->recv_raw.reserve(nk * 4 * W));
    ICD_TRY(g->recv_id.reserve(nk * 8 * W));
    ICD_TRY(g->recv_lv.reserve(nk * W));
    float* s_raw = W == 1 ? (float*)g->recv_raw.ptr : (float*)g->send_raw.ptr;
    int64_t* s_id = W == 1 ? (int64_t*)g->recv_id.ptr : (int64_t*)g->send_id.ptr;
    uint8_t* s_lv = W == 1 ? (uint8_t*)g->recv_lv.ptr : (uint8_t*)g->send_lv.ptr;
    ICD_TRY(index_search_device(x, B, k, local_mode, path, g->row_offset, nullptr, s_raw, s_id, s_lv,
                                q_dtype == ICD_BF16, nullptr, d_mask, st));
    if (W > 1) {
      ICD_NCCL(g_nccl.GroupStart());
      ICD_NCCL(g_nccl.AllGather(s_raw, g->recv_raw.ptr, nk * 4, /*ncclInt8*/ 0, g->comm, st));
      ICD_NCCL(g_nccl.AllGather(s_id, g->recv_id.ptr, nk * 8, 0, g->comm, st));
      ICD_NCCL(g_nccl.AllGather(s_lv, g->recv_lv.ptr, nk, 0, g->comm, st));
      ICD_NCCL(g_nccl.GroupEnd());
    }
    f.cand_score = (const float*)g->recv_raw.ptr;
    f.cand_id = (const int64_t*)g->recv_id.ptr;
    f.cand_level = (const uint8_t*)g->recv_lv.ptr;
    ICD_TRY(launch_finalise(f, st));
  } else {
    // fused peer-store exchange
    SlabLayout L(W);
    g->epoch += 1;
    const int parity = (int)(g->epoch & 1);
    PushTargets push{};
    push.n = W;
    for (int r = 0; r < W; ++r) {
      char* blk = g->peer_slab[r] + L.block(parity, g->rank);
      push.raw[r] = (float*)(blk + L.blk_raw);
      push.id[r] = (int64_t*)(blk + L.blk_id);
      push.level[r] = (uint8_t*)(blk + L.blk_lv);
      push.flag[r] = (uint32_t*)(blk + L.blk_flag);
    }
    push.epoch = g->epoch;
    ICD_TRY(index_search_device(x, B, k, local_mode, path, g->row_offset, nullptr, nullptr, nullptr, nullptr,
                                q_dtype == ICD_BF16, &push, d_mask, st));
    // consumer: sources are the blocks [parity][0..W) of the local slab; fields are strided by block
    char* base = g->slab + L.block(parity, 0);
    f.cand_score = (const float*)(base + L.blk_raw);
    f.cand_id = (const int64_t*)(base + L.blk_id);
    f.cand_level = (const uint8_t*)(base + L.blk_lv);
    f.wait_flag = (const uint32_t*)(base + L.blk_flag);
    f.src_stride_bytes = L.blk_total;
    f.epoch = g->epoch;
    ICD_TRY(launch_finalise(f, st));
  }
  ICD_TRY(copy_out(out_score, k_score, nk * 4, st));
  ICD_TRY(copy_out(out_raw, k_raw, nk * 4, st));
  ICD_TRY(copy_out(out_id, k_id, nk * 8, st));
  const bool host_out = (out_score && !is_device_ptr(out_score)) || (out_raw && !is_device_ptr(out_raw)) ||
                        (out_id && !is_device_ptr(out_id));
  if (sync || host_out || !is_device_ptr(q)) ICD_CUDA(cudaStreamSynchronize(st));
  return ICD_OK;
}

}  // extern "C"
