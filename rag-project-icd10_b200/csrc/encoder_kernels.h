// encoder_kernels.h -- launch interfaces of the BERT encoder kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace icd {

// 1 (default): the kernels of one encoder forward are chained with programmatic dependent launch, so that the prologue of
// kernel i+1 overlaps the tail of kernel i (what a batch-1 forward of 63 small launches is made of); icd_tune("enc_pdl", 0)
// restores plain stream order.  Results never depend on it.
int encoder_pdl();
void encoder_set_pdl(int on);

// cudaLaunchKernelEx with the programmatic-stream-serialization attribute (plus a cluster of `cluster` CTAs when > 1)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster,
                                  Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (encoder_pdl()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = (unsigned)n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

enum GemmEpilogue { EPI_BIAS = 0, EPI_BIAS_GELU = 1, EPI_BIAS_RESIDUAL = 2 };

// Hidden sizes: every launcher whose kernel depends on the width takes it as a trailing `hidden` argument (or struct
// member) that defaults to 768; 768 (BERT-base) and 1024 (BERT-large, XLM-R-large) are instantiated, heads are 64 wide.

// ---- gemm_tc.cu : out[M,N] = epi(A[M,K] * W[N,K]^T + bias)
struct GemmArgs {
  const void* tmap_a;  // 128-byte CUtensorMap of A (box 128 x 64, SWIZZLE_128B)
  const void* tmap_b;  // CUtensorMap of W (box 256 x 64, SWIZZLE_128B)
  const float* bias;   // [N] fp32
  const void* tmap_res;  // CUtensorMap of the residual [rows,N] bf16 (box 128 x 64; EPI_BIAS_RESIDUAL) or null
  const void* tmap_out;  // CUtensorMap of out [rows,N] bf16 (box 128 x 64); rows is a multiple of 128 >= M
  int M, N, K;
  int epi;
  // deferred LayerNorm (gemm_tc.cu header); all optional
  const float* vec2 = nullptr;      // [N] fp32: c = row sums of the gamma-folded W (A is a pre-LN stream), or gamma (residual is one)
  const void* stats_in = nullptr;   // [stats_cols / 128][stats_stride] float2 partial (sum, sum sq) per row of that stream
  void* stats_out = nullptr;        // [N / 128][stats_stride] float2 partials of this GEMM's output rows
  int stats_stride = 0;             // rows per slot, a multiple of 256 >= M
  int stats_cols = 0;               // row length the incoming statistics cover (the hidden size: 768 or 1024)
  float eps = 0.0f;
};
int gemm_tile_n();
int launch_gemm_tc(const GemmArgs& a, cudaStream_t st);
int gemm_make_map_a(void* map128, const void* base, int64_t rows, int K);
int gemm_make_map_b(void* map128, const void* base, int64_t rows, int K);
int gemm_make_map_out(void* map128, const void* base, int64_t rows, int N);

// ---- skinny_linear.cu : the same linear layers for M <= 64 tokens (batch-1 encode_query) on every SM at once
struct SkinnyArgs {
  const void* A;       // [M, K] bf16
  const void* W;       // [N, K] bf16
  const float* bias;   // [N]
  const float* vec2;   // [N]: c when lnin, gamma when the residual goes through a LayerNorm, else null
  const void* res;     // [M, N] bf16 residual stream (EPI_BIAS_RESIDUAL) or null
  void* out;           // [M, N] bf16
  int M, N, K;
  int epi;             // GemmEpilogue
  int lnin;            // A is an un-normalised stream: LayerNorm folded into W / bias / vec2 (rows of `hidden`)
  float eps;
  int hidden = 768;    // row length the LayerNorm statistics cover (768 or 1024)
};
// 1 (default): forwards of at most 64 tokens take this path; icd_tune("enc_skinny", 0) sends them through the tile
// kernels like every larger batch (2 = everything the kernel supports: the same today).  Results agree to bf16 rounding
// (different summation order).  skinny_max_tokens() = the current limit (0 or 64).
int encoder_skinny();
void encoder_set_skinny(int mode);
int skinny_max_tokens();
bool skinny_linear_supported(int M, int N, int K, int hidden = 768);
int launch_skinny_linear(const SkinnyArgs& a, cudaStream_t st);

// ---- encoder_kernels.cu
// h0[M,H] = LayerNorm(word[ids] + pos[pos_offset + t] + type[0]); ids outside [0, vocab) read row `unk`.  pos_offset is
// 0 for BERT and pad_token_id + 1 (= 2) for XLM-R, which numbers the real tokens of a right-padded sequence from there
int launch_embed_ln(const int32_t* ids, int M, int S, int vocab, int unk, const float* word, const float* pos,
                    const float* type0, const float* gamma, const float* beta, float eps, void* out_bf16, cudaStream_t st,
                    int pos_offset = 0, int hidden = 768);
// out = LayerNorm(x) row-wise over H columns
int launch_layernorm(const void* x_bf16, int M, const float* gamma, const float* beta, float eps, void* out_bf16,
                     cudaStream_t st, int hidden = 768);
// attention_tc.cu: softmax(Q K^T / 8 + mask) V for every (sequence, head) on tensor cores (tcgen05); qkv is
// [M, 3H] = [q | k | v]; tmap_qkv from attention_make_map over the [rows, 3H] buffer; H / 64 heads
int attention_make_map(void* map128, const void* qkv_bf16, int64_t rows, int hidden = 768);
// ctx_rows = rows of the ctx buffer (a multiple of 128 >= B*S): the store boxes are clipped against it
int launch_attention_tc(const void* tmap_qkv, const int32_t* lens, int B, int S, void* ctx_bf16, int64_t ctx_rows,
                        cudaStream_t st, int hidden = 768);
// the same for 128 < S <= 512 (token-classification path) on the same tensor-core kernel in split-KV mode: one item per
// (sequence, head, query tile, key tile), partial outputs + row statistics into scratch, then a combine kernel
size_t attention_long_scratch_bytes(int B, int S, size_t* stats_bytes, int hidden = 768);
int launch_attention_tc_long(const void* tmap_qkv, const int32_t* lens, int B, int S, void* part_scratch, void* stats_scratch,
                             void* ctx_bf16, cudaStream_t st, int hidden = 768);
// masked mean over tokens + L2 normalise -> [B,H] (fp32 or bf16)
int launch_pool_normalise(const void* h_bf16, const int32_t* lens, int B, int S, void* out, int out_dtype,
                          cudaStream_t st, int hidden = 768);

// logits[m, l] = h[m, :] . w[l, :] + b[l]  (h bf16 [M, H], w fp32 [L, H], out fp32 [M, L]); L <= 64
int launch_token_head(const void* h_bf16, int M, const float* w, const float* b, int L, float* out, cudaStream_t st,
                      int hidden = 768);

}  // namespace icd
