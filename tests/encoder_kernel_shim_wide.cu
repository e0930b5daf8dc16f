// encoder_kernel_shim_wide.cu -- test-only extern "C" entries over the encoder launchers of libicdrag.so, with the
// hidden size as an argument (768 or 1024).
//
// tests/test_wide_encoder_gpu.py compiles this file into its temporary directory, links it against the shipped
// csrc/libicdrag.so and loads it with ctypes, as tests/test_encoder_kernels_gpu.py does with encoder_kernel_shim.cu
// (which calls every launcher with its default width, 768).  Each entry takes device pointers and a stream, builds the
// tensor maps through the library's own icd::*_make_map_* functions and returns the launcher's status.  Nothing here
// allocates, copies or synchronises.
#include "encoder_kernels.h"
#include "icdrag.h"
#include "kernels.h"

using namespace icd;

extern "C" {

// out[M, N] = epi(A W^T + bias); stats_cols = the hidden size the incoming statistics cover
int wshim_gemm(const void* A, long a_rows, const void* W, const float* bias, const float* vec2, const void* res,
               void* out, long out_rows, int M, int N, int K, int epi, const void* stats_in, void* stats_out,
               int stats_stride, int stats_cols, float eps, void* stream) {
  alignas(128) unsigned char ma[128], mb[128], mo[128], mr[128];
  int st = gemm_make_map_a(ma, A, a_rows, K);
  if (st == ICD_OK) st = gemm_make_map_b(mb, W, N, K);
  if (st == ICD_OK) st = gemm_make_map_out(mo, out, out_rows, N);
  if (st == ICD_OK && res) st = gemm_make_map_out(mr, res, out_rows, N);
  if (st != ICD_OK) return st;
  GemmArgs g{};
  g.tmap_a = ma;
  g.tmap_b = mb;
  g.bias = bias;
  g.tmap_res = res ? mr : nullptr;
  g.tmap_out = mo;
  g.M = M, g.N = N, g.K = K;
  g.epi = epi;
  g.vec2 = vec2;
  g.stats_in = stats_in;
  g.stats_out = stats_out;
  g.stats_stride = stats_stride;
  g.stats_cols = stats_cols;
  g.eps = eps;
  return launch_gemm_tc(g, static_cast<cudaStream_t>(stream));
}

int wshim_skinny_supported(int M, int N, int K, int hidden) { return skinny_linear_supported(M, N, K, hidden) ? 1 : 0; }

int wshim_skinny(const void* A, const void* W, const float* bias, const float* vec2, const void* res, void* out, int M,
                 int N, int K, int epi, int lnin, float eps, int hidden, void* stream) {
  SkinnyArgs s{A, W, bias, vec2, res, out, M, N, K, epi, lnin, eps, hidden};
  return launch_skinny_linear(s, static_cast<cudaStream_t>(stream));
}

int wshim_attention(const void* qkv, long qkv_rows, const int32_t* lens, int B, int S, void* ctx, long ctx_rows,
                    int hidden, void* stream) {
  alignas(128) unsigned char mq[128];
  const int st = attention_make_map(mq, qkv, qkv_rows, hidden);
  if (st != ICD_OK) return st;
  return launch_attention_tc(mq, lens, B, S, ctx, ctx_rows, static_cast<cudaStream_t>(stream), hidden);
}

long wshim_attention_long_scratch(int B, int S, int hidden, long* stats_bytes) {
  size_t sb = 0;
  const size_t pb = attention_long_scratch_bytes(B, S, &sb, hidden);
  *stats_bytes = (long)sb;
  return (long)pb;
}

int wshim_attention_long(const void* qkv, long qkv_rows, const int32_t* lens, int B, int S, void* part, void* stats,
                         void* ctx, int hidden, void* stream) {
  alignas(128) unsigned char mq[128];
  const int st = attention_make_map(mq, qkv, qkv_rows, hidden);
  if (st != ICD_OK) return st;
  return launch_attention_tc_long(mq, lens, B, S, part, stats, ctx, static_cast<cudaStream_t>(stream), hidden);
}

int wshim_embed_ln(const int32_t* ids, int M, int S, int vocab, int unk, const float* word, const float* pos,
                   const float* type0, const float* gamma, const float* beta, float eps, void* out, int pos_offset,
                   int hidden, void* stream) {
  return launch_embed_ln(ids, M, S, vocab, unk, word, pos, type0, gamma, beta, eps, out, static_cast<cudaStream_t>(stream),
                         pos_offset, hidden);
}

int wshim_layernorm(const void* x, int M, const float* gamma, const float* beta, float eps, void* out, int hidden,
                    void* stream) {
  return launch_layernorm(x, M, gamma, beta, eps, out, static_cast<cudaStream_t>(stream), hidden);
}

int wshim_pool_normalise(const void* h, const int32_t* lens, int B, int S, void* out, int out_dtype, int hidden,
                         void* stream) {
  return launch_pool_normalise(h, lens, B, S, out, out_dtype, static_cast<cudaStream_t>(stream), hidden);
}

int wshim_token_head(const void* h, int M, const float* w, const float* b, int L, float* out, int hidden, void* stream) {
  return launch_token_head(h, M, w, b, L, out, static_cast<cudaStream_t>(stream), hidden);
}

}  // extern "C"
