// encoder_kernels.cu -- the memory-bound pieces of the BERT encoder around the tcgen05 GEMMs:
// embedding gather + LayerNorm, LayerNorm, small-sequence attention, masked mean pool + L2
// normalise.  Arithmetic follows transformers.BertModel as driven by
// SentenceTransformer.encode (reference call sites services/embedding_service.py:81,97,120).
// Hidden size H is a template parameter, instantiated for 768 (BERT-base) and 1024 (BERT-large, XLM-R-large): a warp per
// token holds H / 32 elements per lane (24 or 32, H / 256 chunks of 8); heads of 64.
#include "common.cuh"
#include "encoder_kernels.h"
#include "ptx.cuh"

namespace icd {
namespace {


__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// lane owns elements c*256 + lane*8 + e  (c = 0..H/256-1, e = 0..7): 16-byte bf16 accesses, coalesced
template <int H>
__device__ __forceinline__ void ln_store(const float* x, const float* __restrict__ gamma,
                                         const float* __restrict__ beta, float eps, __nv_bfloat16* out_row, int lane) {
  constexpr int kPerLane = H / 32;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kPerLane; ++i) s += x[i];
  const float mean = warp_sum(s) * (1.0f / H);
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < kPerLane; ++i) {
    const float d = x[i] - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = rsqrtf(warp_sum(v) * (1.0f / H) + eps);
#pragma unroll
  for (int c = 0; c < H / 256; ++c) {
    const int col = c * 256 + lane * 8;
    const float4 g0 = *reinterpret_cast<const float4*>(gamma + col), g1 = *reinterpret_cast<const float4*>(gamma + col + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(beta + col), b1 = *reinterpret_cast<const float4*>(beta + col + 4);
    const float* xx = x + c * 8;
    uint4 o;
    o.x = pack2((xx[0] - mean) * rstd * g0.x + b0.x, (xx[1] - mean) * rstd * g0.y + b0.y);
    o.y = pack2((xx[2] - mean) * rstd * g0.z + b0.z, (xx[3] - mean) * rstd * g0.w + b0.w);
    o.z = pack2((xx[4] - mean) * rstd * g1.x + b1.x, (xx[5] - mean) * rstd * g1.y + b1.y);
    o.w = pack2((xx[6] - mean) * rstd * g1.z + b1.z, (xx[7] - mean) * rstd * g1.w + b1.w);
    *reinterpret_cast<uint4*>(out_row + col) = o;
  }
}

// position of token t of a sequence: pos_offset + t (0 for BERT; XLM-R numbers real tokens from pad_token_id + 1 = 2)
template <int H>
__global__ void __launch_bounds__(256)
embed_ln_kernel(const int32_t* __restrict__ ids, int M, int S, int vocab, int unk, int pos_offset,
                const float* __restrict__ word, const float* __restrict__ pos, const float* __restrict__ type0,
                const float* __restrict__ gamma, const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ out) {
  ptx::griddep_launch();
  ptx::griddep_wait();   // `out` is read by kernels of the previous forward that may still be running
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tok = blockIdx.x * 8 + warp;
  if (tok >= M) return;
  int id = ids[tok];
  if ((unsigned)id >= (unsigned)vocab) id = unk;  // an id outside the table (mismatched vocab.txt) reads [UNK], not foreign memory
  const int t = tok % S + pos_offset;
  float x[H / 32];
#pragma unroll
  for (int c = 0; c < H / 256; ++c) {
    const int col = c * 256 + lane * 8;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const float4 w = *reinterpret_cast<const float4*>(word + (size_t)id * H + col + 4 * h);
      const float4 p = *reinterpret_cast<const float4*>(pos + (size_t)t * H + col + 4 * h);
      const float4 ty = *reinterpret_cast<const float4*>(type0 + col + 4 * h);
      x[c * 8 + 4 * h + 0] = w.x + ty.x + p.x;
      x[c * 8 + 4 * h + 1] = w.y + ty.y + p.y;
      x[c * 8 + 4 * h + 2] = w.z + ty.z + p.z;
      x[c * 8 + 4 * h + 3] = w.w + ty.w + p.w;
    }
  }
  ln_store<H>(x, gamma, beta, eps, out + (size_t)tok * H, lane);
}

template <int H>
__global__ void __launch_bounds__(256)
layernorm_kernel(const __nv_bfloat16* __restrict__ in, int M, const float* __restrict__ gamma,
                 const float* __restrict__ beta, float eps, __nv_bfloat16* __restrict__ out) {
  ptx::griddep_launch();
  ptx::griddep_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tok = blockIdx.x * 8 + warp;
  if (tok >= M) return;
  float x[H / 32];
#pragma unroll
  for (int c = 0; c < H / 256; ++c) {
    const uint4 v = *reinterpret_cast<const uint4*>(in + (size_t)tok * H + c * 256 + lane * 8);
    x[c * 8 + 0] = bf16lo_to_f32(v.x);
    x[c * 8 + 1] = bf16hi_to_f32(v.x);
    x[c * 8 + 2] = bf16lo_to_f32(v.y);
    x[c * 8 + 3] = bf16hi_to_f32(v.y);
    x[c * 8 + 4] = bf16lo_to_f32(v.z);
    x[c * 8 + 5] = bf16hi_to_f32(v.z);
    x[c * 8 + 6] = bf16lo_to_f32(v.w);
    x[c * 8 + 7] = bf16hi_to_f32(v.w);
  }
  ln_store<H>(x, gamma, beta, eps, out + (size_t)tok * H, lane);
}

// ---------------------------------------------------------------- masked mean + L2 normalise
// sentence-transformers Pooling(mean) + F.normalize: sum(h*mask)/clamp(sum(mask),1e-9), then
// x / max(||x||, 1e-12).  One CTA (256 threads, H / 256 columns each) per sequence.
template <int H>
__global__ void __launch_bounds__(256)
pool_normalise_kernel(const __nv_bfloat16* __restrict__ h, const int32_t* __restrict__ lens, int S,
                      void* __restrict__ out, int out_dtype, int normalise) {
  ptx::griddep_launch();
  ptx::griddep_wait();
  __shared__ float red[8];
  const int b = blockIdx.x;
  const int len = min(lens[b], S);
  constexpr int kCols = H / 256;
  float acc[kCols];
#pragma unroll
  for (int c = 0; c < kCols; ++c) acc[c] = 0.f;
  for (int t = 0; t < len; ++t) {
    const __nv_bfloat16* row = h + ((size_t)b * S + t) * H;
#pragma unroll
    for (int c = 0; c < kCols; ++c) acc[c] += __bfloat162float(row[c * 256 + threadIdx.x]);
  }
  const float denom = fmaxf((float)len, 1e-9f);
  float ss = 0.f;
#pragma unroll
  for (int c = 0; c < kCols; ++c) {
    acc[c] /= denom;
    ss = fmaf(acc[c], acc[c], ss);
  }
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += red[w];
  const float inv = normalise ? 1.0f / fmaxf(sqrtf(tot), 1e-12f) : 1.0f;
#pragma unroll
  for (int c = 0; c < kCols; ++c) {
    const float v = acc[c] * inv;
    const size_t o = (size_t)b * H + c * 256 + threadIdx.x;
    if (out_dtype == ICD_F32)
      reinterpret_cast<float*>(out)[o] = v;
    else
      reinterpret_cast<__nv_bfloat16*>(out)[o] = __float2bfloat16_rn(v);
  }
}

// Token-classification head (BertForTokenClassification.classifier): one warp per token row.  The row (H bf16)
// sits in registers, H / 32 elements per lane; the L weight rows stream from L1/L2 (the same 3 / 4 KiB rows for every
// warp) as coalesced fp32 and each label costs one warp reduction.  HBM-bound on the hidden states (2 H bytes per
// token in, 4 L bytes out).
template <int H>
__global__ void __launch_bounds__(256)
token_head_kernel(const __nv_bfloat16* __restrict__ h, int M, const float* __restrict__ w,
                  const float* __restrict__ b, int L, float* __restrict__ out) {
  ptx::griddep_launch();
  ptx::griddep_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  constexpr int kPerLane = H / 32;
  float x[kPerLane];
  const __nv_bfloat16* row = h + (size_t)m * H;
#pragma unroll
  for (int j = 0; j < kPerLane; ++j) x[j] = __bfloat162float(row[j * 32 + lane]);
  for (int l = 0; l < L; ++l) {
    const float* wr = w + (size_t)l * H;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < kPerLane; ++j) acc = fmaf(x[j], __ldg(wr + j * 32 + lane), acc);
    acc = warp_sum(acc);
    if (lane == 0) out[(size_t)m * L + l] = acc + __ldg(b + l);
  }
}

}  // namespace

static int g_encoder_pdl = 1;  // validated in r02o: parity suite green, batch-1 forward 0.85 -> 0.72 ms
int encoder_pdl() { return g_encoder_pdl; }
void encoder_set_pdl(int on) { g_encoder_pdl = on ? 1 : 0; }

static bool supported_hidden(int hidden, const char* who) {
  if (hidden == 768 || hidden == 1024) return true;
  set_error("%s: hidden size %d is not supported (768 or 1024)", who, hidden);
  return false;
}

int launch_token_head(const void* h, int M, const float* w, const float* b, int L, float* out, cudaStream_t st, int hidden) {
  if (!supported_hidden(hidden, "token_head")) return ICD_E_ARG;
  if (M <= 0) return ICD_OK;
  ICD_CUDA(launch_chained(hidden == 768 ? token_head_kernel<768> : token_head_kernel<1024>, dim3((M + 7) / 8), dim3(256), 0, st, 1,
                          reinterpret_cast<const __nv_bfloat16*>(h), M, w, b, L, out));
  count_launch();
  return ICD_OK;
}

int launch_embed_ln(const int32_t* ids, int M, int S, int vocab, int unk, const float* word, const float* pos,
                    const float* type0, const float* gamma, const float* beta, float eps, void* out, cudaStream_t st,
                    int pos_offset, int hidden) {
  if (!supported_hidden(hidden, "embed_ln")) return ICD_E_ARG;
  ICD_CUDA(launch_chained(hidden == 768 ? embed_ln_kernel<768> : embed_ln_kernel<1024>, dim3((M + 7) / 8), dim3(256), 0, st, 1, ids, M,
                          S, vocab, unk, pos_offset, word, pos, type0, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(out)));
  count_launch();
  return ICD_OK;
}

int launch_layernorm(const void* x, int M, const float* gamma, const float* beta, float eps, void* out,
                     cudaStream_t st, int hidden) {
  if (!supported_hidden(hidden, "layernorm")) return ICD_E_ARG;
  ICD_CUDA(launch_chained(hidden == 768 ? layernorm_kernel<768> : layernorm_kernel<1024>, dim3((M + 7) / 8), dim3(256), 0, st, 1,
                          reinterpret_cast<const __nv_bfloat16*>(x), M, gamma, beta, eps, reinterpret_cast<__nv_bfloat16*>(out)));
  count_launch();
  return ICD_OK;
}

int launch_pool_normalise(const void* h, const int32_t* lens, int B, int S, void* out, int out_dtype,
                          cudaStream_t st, int hidden) {
  if (!supported_hidden(hidden, "pool_normalise")) return ICD_E_ARG;
  ICD_CUDA(launch_chained(hidden == 768 ? pool_normalise_kernel<768> : pool_normalise_kernel<1024>, dim3(B), dim3(256), 0, st, 1,
                          reinterpret_cast<const __nv_bfloat16*>(h), lens, S, out, out_dtype & 0xff,
                          (out_dtype & ICD_OUT_NO_NORMALISE) ? 0 : 1));
  count_launch();
  return ICD_OK;
}

}  // namespace icd
