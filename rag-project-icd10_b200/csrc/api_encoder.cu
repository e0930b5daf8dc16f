// api_encoder.cu -- C ABI of the BERT sentence encoder (include/icdrag.h, icd_encoder_*).
//
// Stands where SentenceTransformer(...).encode(normalize_embeddings=True) stands in the
// reference (services/embedding_service.py:61,81,97-102,120).  Two shapes: hidden 768 / 12 heads (BERT-base) and
// hidden 1024 / 16 heads (BERT-large, XLM-R-large: the reference's default intfloat/multilingual-e5-large-instruct);
// XLM-R is the same post-LN encoder with its positions numbered from pad_token_id + 1 and <unk> = 3
// (icd_encoder_set_embedding_ids).  Weight blob order (fp32, HF BertModel names; XLMRobertaModel has the same ones)
// -- mirrored by rag-project-icd10_b200/engine/weights.py:
//   embeddings.word_embeddings.weight        [V, H]
//   embeddings.position_embeddings.weight    [P, H]
//   embeddings.token_type_embeddings.weight  [T, H]
//   embeddings.LayerNorm.weight / .bias      [H] [H]
//   per layer l:
//     attention.self.query.weight, key.weight, value.weight      3 x [H, H]
//     attention.self.query.bias, key.bias, value.bias            3 x [H]
//     attention.output.dense.weight [H, H], .bias [H]
//     attention.output.LayerNorm.weight / .bias                  [H] [H]
//     intermediate.dense.weight [I, H], .bias [I]
//     output.dense.weight [H, I], .bias [H]
//     output.LayerNorm.weight / .bias                            [H] [H]
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "encoder_kernels.h"
#include "kernels.h"

namespace icd {

struct LayerW {
  // bf16 GEMM weights ([out, in] row-major == K-major B operand) and their TMA maps
  void *wqkv, *wo, *w1, *w2;
  alignas(128) unsigned char m_qkv[128];
  alignas(128) unsigned char m_o[128];
  alignas(128) unsigned char m_1[128];
  alignas(128) unsigned char m_2[128];
  // fp32 small parameters
  float *bqkv, *bo, *ln1g, *ln1b, *b1, *b2, *ln2g, *ln2b;
  // deferred-LayerNorm mode (gemm_tc.cu header): wqkv / w1 hold W diag(gamma) of the LayerNorm in front of them,
  // bqkv / b1 the matching b + W beta, cqkv / c1 the row sums of the folded bf16 weights (null: input is already
  // normalised, layer 0's QKV), bo_r / b2_r the bias plus the beta of the LayerNorm the residual goes through
  float *cqkv = nullptr, *c1 = nullptr, *bo_r = nullptr, *b2_r = nullptr;
};

}  // namespace icd

struct icd_encoder {
  icd_bert_cfg cfg;
  int device = 0;
  // fp32 embedding tables and LN
  float *word = nullptr, *pos = nullptr, *type = nullptr, *eg = nullptr, *eb = nullptr;
  std::vector<icd::LayerW*> layers;
  std::vector<void*> allocs;
  // activations (bf16) for max_tokens rows
  int max_tokens = 0;
  void *h = nullptr, *h1 = nullptr, *t = nullptr, *ctx = nullptr, *qkv = nullptr, *f = nullptr;
  alignas(128) unsigned char m_h[128];
  alignas(128) unsigned char m_h1[128];
  alignas(128) unsigned char m_ctx[128];
  alignas(128) unsigned char m_f[128];
  alignas(128) unsigned char m_qkv[128];
  alignas(128) unsigned char m_t[128];        // GEMM output maps (box 128 x 64)
  alignas(128) unsigned char m_qkv_out[128];
  // deferred LayerNorm: per-row partial (sum, sum sq) of the two pre-LayerNorm streams, [H/128][stats_stride] float2
  bool fused_ln = true;
  void *stats1 = nullptr, *stats2 = nullptr;
  int stats_stride = 0;
  int32_t *ids = nullptr, *lens = nullptr;
  int ids_cap = 0, lens_cap = 0;
  void* out_stage = nullptr;
  size_t out_cap = 0;
  // scratch of the split-KV attention (sequences beyond 128 tokens): partial outputs and row statistics
  void *att_part = nullptr, *att_stats = nullptr;
  size_t att_part_cap = 0, att_stats_cap = 0;
  int last_M = 0;
  // token-classification head (icd_encoder_set_token_head): logits = h W^T + b per token
  float *head_w = nullptr, *head_b = nullptr;
  int head_labels = 0;
  // icd_encoder_set_embedding_ids: token t of a sequence reads position row pos_offset + t; ids outside the table read unk
  int pos_offset = 0;
  int unk = 0;
};

namespace icd {

static int64_t weight_count(const icd_bert_cfg& c) {
  const int64_t H = c.hidden, I = c.intermediate;
  int64_t n = (int64_t)c.vocab_size * H + (int64_t)c.max_position * H + (int64_t)c.type_vocab * H + 2 * H;
  n += (int64_t)c.layers * (3 * H * H + 3 * H + H * H + H + 2 * H + I * H + I + H * I + H + 2 * H);
  return n;
}

// ids outside the embedding table read [UNK] (100 in BERT vocabularies) unless icd_encoder_set_embedding_ids says otherwise
static int default_unk(const icd_bert_cfg& c) { return c.vocab_size > 100 ? 100 : 0; }

static int dev_alloc(icd_encoder* e, void** p, size_t bytes) {
  ICD_CUDA(cudaMalloc(p, bytes));
  e->allocs.push_back(*p);
  return ICD_OK;
}

// upload `n` fp32 values from host `src` as fp32 (keep) or bf16 (GEMM weights)
static int upload(icd_encoder* e, const float* src, int64_t n, bool as_bf16, void** out, float* stage) {
  if (!as_bf16) {
    ICD_TRY(dev_alloc(e, out, (size_t)n * 4));
    ICD_CUDA(cudaMemcpy(*out, src, (size_t)n * 4, cudaMemcpyDefault));
    return ICD_OK;
  }
  ICD_TRY(dev_alloc(e, out, (size_t)n * 2));
  ICD_CUDA(cudaMemcpy(stage, src, (size_t)n * 4, cudaMemcpyDefault));
  ICD_TRY(launch_f32_to_bf16(stage, *out, n, 0));
  ICD_CUDA(cudaStreamSynchronize(0));
  return ICD_OK;
}

static int reserve_tokens(icd_encoder* e, int max_tokens) {
  if (max_tokens <= e->max_tokens) return ICD_OK;
  const int H = e->cfg.hidden, I = e->cfg.intermediate;
  const int M = ((max_tokens + 127) / 128) * 128;
  void** bufs[6] = {&e->h, &e->h1, &e->t, &e->ctx, &e->qkv, &e->f};
  const size_t widths[6] = {(size_t)H, (size_t)H, (size_t)H, (size_t)H, (size_t)3 * H, (size_t)I};
  for (int i = 0; i < 6; ++i) {
    if (*bufs[i]) cudaFree(*bufs[i]);
    *bufs[i] = nullptr;
  }
  if (e->stats1) cudaFree(e->stats1);
  if (e->stats2) cudaFree(e->stats2);
  e->stats1 = e->stats2 = nullptr;
  e->max_tokens = 0;
  for (int i = 0; i < 6; ++i) {
    ICD_CUDA(cudaMalloc(bufs[i], (size_t)M * widths[i] * 2));
    ICD_CUDA(cudaMemset(*bufs[i], 0, (size_t)M * widths[i] * 2));
  }
  // a CTA pair's tile is 256 rows: the statistics rows cover whole tiles
  e->stats_stride = ((M + 255) / 256) * 256;
  const size_t stats_bytes = (size_t)(H / 128) * e->stats_stride * 8;
  ICD_CUDA(cudaMalloc(&e->stats1, stats_bytes));
  ICD_CUDA(cudaMalloc(&e->stats2, stats_bytes));
  ICD_CUDA(cudaMemset(e->stats1, 0, stats_bytes));
  ICD_CUDA(cudaMemset(e->stats2, 0, stats_bytes));
  ICD_TRY(gemm_make_map_a(e->m_h, e->h, M, H));
  ICD_TRY(gemm_make_map_a(e->m_h1, e->h1, M, H));
  ICD_TRY(gemm_make_map_a(e->m_ctx, e->ctx, M, H));
  ICD_TRY(gemm_make_map_a(e->m_f, e->f, M, I));
  ICD_TRY(attention_make_map(e->m_qkv, e->qkv, M, H));
  ICD_TRY(gemm_make_map_out(e->m_t, e->t, M, H));
  ICD_TRY(gemm_make_map_out(e->m_qkv_out, e->qkv, M, 3 * H));
  e->max_tokens = M;
  return ICD_OK;
}

// round-to-nearest-even fp32 -> bf16 -> fp32, the rounding f32_to_bf16_kernel applies on the device
static float bf16_round_host(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  u += 0x7fffu + ((u >> 16) & 1u);
  u &= 0xffff0000u;
  memcpy(&f, &u, 4);
  return f;
}

// Folds the LayerNorm (gamma, beta) in front of a linear layer y = LN(x) W^T + b into the layer:
//   wf[n,k] = W[n,k] gamma[k];  bf[n] = b[n] + sum_k W[n,k] beta[k];  c[n] = sum_k bf16(wf[n,k])
// so that y = rs (x wf^T) - rs mu c + bf with the row statistics applied in the GEMM epilogue.
static void fold_layernorm(const float* W, const float* b, const float* gamma, const float* beta, int64_t n_out,
                           int64_t n_in, std::vector<float>& wf, std::vector<float>& bf, std::vector<float>& c) {
  wf.resize((size_t)n_out * n_in);
  bf.resize((size_t)n_out);
  c.resize((size_t)n_out);
  for (int64_t n = 0; n < n_out; ++n) {
    double bacc = b[n], cacc = 0.0;
    const float* w = W + n * n_in;
    float* o = wf.data() + n * n_in;
    for (int64_t k = 0; k < n_in; ++k) {
      o[k] = w[k] * gamma[k];
      cacc += (double)bf16_round_host(o[k]);
      bacc += (double)w[k] * (double)beta[k];
    }
    bf[n] = (float)bacc;
    c[n] = (float)cacc;
  }
}

}  // namespace icd

using namespace icd;

extern "C" {

int64_t icd_encoder_weight_count(const icd_bert_cfg* cfg) { return cfg ? weight_count(*cfg) : -1; }

int icd_encoder_create(const float* weights, int64_t count, const icd_bert_cfg* cfg, int device, icd_encoder** out) {
  ICD_CHECK_ARG(weights && cfg && out, "null argument");
  ICD_CHECK_ARG((cfg->hidden == 768 && cfg->heads == 12) || (cfg->hidden == 1024 && cfg->heads == 16),
                "supported shapes are hidden=768 with heads=12 and hidden=1024 with heads=16 (head dim 64)");
  ICD_CHECK_ARG(cfg->intermediate > 0 && cfg->intermediate % gemm_tile_n() == 0, "intermediate must be a multiple of 256");
  ICD_CHECK_ARG(cfg->layers >= 1 && cfg->vocab_size > 0 && cfg->max_position > 0 && cfg->type_vocab > 0, "bad config");
  ICD_CHECK_ARG(count == weight_count(*cfg), "weight blob size does not match the config");
  int ndev = 0;
  ICD_CUDA(cudaGetDeviceCount(&ndev));
  ICD_CHECK_ARG(device >= 0 && device < ndev, "no such CUDA device");
  ICD_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  ICD_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    set_error("libicdrag is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    return ICD_E_UNSUPPORTED;
  }
  icd_encoder* e = new icd_encoder();
  e->cfg = *cfg;
  e->device = device;
  e->unk = default_unk(*cfg);
  const int64_t H = cfg->hidden, I = cfg->intermediate;
  float* stage = nullptr;
  const int64_t stage_n = std::max<int64_t>(3 * H * H, I * H);
  int st = ICD_OK;
  auto fail = [&](int s) {
    if (stage) cudaFree(stage);
    icd_encoder_destroy(e);
    return s;
  };
  if (cudaMalloc((void**)&stage, (size_t)stage_n * 4) != cudaSuccess) {
    set_error("staging allocation failed");
    return fail(ICD_E_NOMEM);
  }
  const float* w = weights;
  auto take = [&](int64_t n, bool bf16, void** dst) {
    if (st != ICD_OK) return;
    st = upload(e, w, n, bf16, dst, stage);
    w += n;
  };
  take((int64_t)cfg->vocab_size * H, false, (void**)&e->word);
  take((int64_t)cfg->max_position * H, false, (void**)&e->pos);
  take((int64_t)cfg->type_vocab * H, false, (void**)&e->type);
  take(H, false, (void**)&e->eg);
  take(H, false, (void**)&e->eb);
#ifdef ICD_PROFILING
  // profiling builds only: ICD_ENC_FUSED_LN=0 keeps the separate LayerNorm launches (A/B timing)
  {
    const char* v = getenv("ICD_ENC_FUSED_LN");
    e->fused_ln = !(v && *v && atoi(v) == 0);
  }
#endif
  const float *prev_g = nullptr, *prev_b = nullptr;  // host: the LayerNorm that closes the previous layer
  std::vector<float> wf, bf, cf, sum;
  auto upload_vec = [&](const std::vector<float>& v, float** dst) {
    if (st != ICD_OK) return;
    st = upload(e, v.data(), (int64_t)v.size(), false, (void**)dst, stage);
  };
  for (int l = 0; l < cfg->layers && st == ICD_OK; ++l) {
    LayerW* L = new LayerW();
    e->layers.push_back(L);
    const float* h_wqkv = w;
    const float* h_bqkv = h_wqkv + 3 * H * H;
    const float* h_wo = h_bqkv + 3 * H;
    const float* h_bo = h_wo + H * H;
    const float* h_g1 = h_bo + H;
    const float* h_be1 = h_g1 + H;
    const float* h_w1 = h_be1 + H;
    const float* h_b1 = h_w1 + I * H;
    const float* h_w2 = h_b1 + I;
    const float* h_b2 = h_w2 + H * I;
    const float* h_g2 = h_b2 + H;
    const float* h_be2 = h_g2 + H;
    if (e->fused_ln && prev_g) {
      fold_layernorm(h_wqkv, h_bqkv, prev_g, prev_b, 3 * H, H, wf, bf, cf);
      if (st == ICD_OK) st = upload(e, wf.data(), 3 * H * H, true, &L->wqkv, stage);
      upload_vec(bf, &L->bqkv);
      upload_vec(cf, &L->cqkv);
      w += 3 * H * H + 3 * H;
    } else {
      take(3 * H * H, true, &L->wqkv);
      take(3 * H, false, (void**)&L->bqkv);
    }
    take(H * H, true, &L->wo);
    take(H, false, (void**)&L->bo);
    take(H, false, (void**)&L->ln1g);
    take(H, false, (void**)&L->ln1b);
    if (e->fused_ln) {
      fold_layernorm(h_w1, h_b1, h_g1, h_be1, I, H, wf, bf, cf);
      if (st == ICD_OK) st = upload(e, wf.data(), I * H, true, &L->w1, stage);
      upload_vec(bf, &L->b1);
      upload_vec(cf, &L->c1);
      w += I * H + I;
    } else {
      take(I * H, true, &L->w1);
      take(I, false, (void**)&L->b1);
    }
    take(H * I, true, &L->w2);
    take(H, false, (void**)&L->b2);
    take(H, false, (void**)&L->ln2g);
    take(H, false, (void**)&L->ln2b);
    if (e->fused_ln) {
      // the residual epilogues rebuild LN(x) = (x - mu) rs gamma + beta from the stream: beta rides in the bias
      sum.assign(h_bo, h_bo + H);
      if (prev_b)
        for (int64_t i = 0; i < H; ++i) sum[i] += prev_b[i];
      upload_vec(sum, &L->bo_r);
      sum.assign(h_b2, h_b2 + H);
      for (int64_t i = 0; i < H; ++i) sum[i] += h_be1[i];
      upload_vec(sum, &L->b2_r);
    }
    prev_g = h_g2;
    prev_b = h_be2;
    if (st != ICD_OK) break;
    st = gemm_make_map_b(L->m_qkv, L->wqkv, 3 * H, (int)H);
    if (st == ICD_OK) st = gemm_make_map_b(L->m_o, L->wo, H, (int)H);
    if (st == ICD_OK) st = gemm_make_map_b(L->m_1, L->w1, I, (int)H);
    if (st == ICD_OK) st = gemm_make_map_b(L->m_2, L->w2, H, (int)I);
  }
  if (st != ICD_OK) return fail(st);
  cudaFree(stage);
  stage = nullptr;
  *out = e;
  return ICD_OK;
}

int icd_encoder_destroy(icd_encoder* e) {
  if (!e) return ICD_OK;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (void* p : e->allocs) cudaFree(p);
  for (auto* L : e->layers) delete L;
  void* bufs[] = {e->h, e->h1, e->t, e->ctx, e->qkv, e->f, e->ids, e->lens, e->out_stage, e->stats1, e->stats2,
                  e->head_w, e->head_b, e->att_part, e->att_stats};
  for (void* p : bufs)
    if (p) cudaFree(p);
  delete e;
  return ICD_OK;
}

int icd_encoder_reserve(icd_encoder* e, int max_tokens) {
  ICD_CHECK_ARG(e != nullptr && max_tokens > 0, "bad argument");
  ICD_CUDA(cudaSetDevice(e->device));
  return reserve_tokens(e, max_tokens);
}

}  // extern "C"

namespace icd {

// Runs embeddings + all layers for B sequences padded to S; on return *final_h is the [B*S, hidden] bf16 buffer of
// last-layer hidden states and *d_lens_out the device copy of the lengths.  Work is enqueued on st.
static int encode_hidden(icd_encoder* e, const int32_t* ids, const int32_t* lens, int B, int S, cudaStream_t st,
                         const void** final_h_out, const int32_t** d_lens_out) {
  const int M = B * S;
  ICD_TRY(reserve_tokens(e, M));
  const int H = e->cfg.hidden, I = e->cfg.intermediate;
  const float eps = e->cfg.ln_eps;

  // token ids / lengths -> device
  const int32_t* d_ids = ids;
  const int32_t* d_lens = lens;
  if (!is_device_ptr(ids)) {
    if (M > e->ids_cap) {
      if (e->ids) cudaFree(e->ids);
      e->ids = nullptr;
      ICD_CUDA(cudaMalloc((void**)&e->ids, (size_t)M * 4));
      e->ids_cap = M;
    }
    ICD_CUDA(cudaMemcpyAsync(e->ids, ids, (size_t)M * 4, cudaMemcpyHostToDevice, st));
    d_ids = e->ids;
  }
  if (!is_device_ptr(lens)) {
    if (B > e->lens_cap) {
      if (e->lens) cudaFree(e->lens);
      e->lens = nullptr;
      ICD_CUDA(cudaMalloc((void**)&e->lens, (size_t)B * 4));
      e->lens_cap = B;
    }
    ICD_CUDA(cudaMemcpyAsync(e->lens, lens, (size_t)B * 4, cudaMemcpyHostToDevice, st));
    d_lens = e->lens;
  }
  // ids outside the embedding table read the unk row instead of faulting
  ICD_TRY(launch_embed_ln(d_ids, M, S, e->cfg.vocab_size, e->unk, e->word, e->pos, e->type, e->eg, e->eb, eps, e->h, st,
                          e->pos_offset, H));
  if (S > 128) {
    size_t stats_bytes = 0;
    const size_t part_bytes = attention_long_scratch_bytes(B, S, &stats_bytes, H);
    if (part_bytes > e->att_part_cap) {
      if (e->att_part) cudaFree(e->att_part);
      e->att_part = nullptr, e->att_part_cap = 0;
      ICD_CUDA(cudaMalloc(&e->att_part, part_bytes));
      e->att_part_cap = part_bytes;
    }
    if (stats_bytes > e->att_stats_cap) {
      if (e->att_stats) cudaFree(e->att_stats);
      e->att_stats = nullptr, e->att_stats_cap = 0;
      ICD_CUDA(cudaMalloc(&e->att_stats, stats_bytes));
      e->att_stats_cap = stats_bytes;
    }
  }
  auto attention = [&]() {
    return S <= 128 ? launch_attention_tc(e->m_qkv, d_lens, B, S, e->ctx, e->max_tokens, st, H)
                    : launch_attention_tc_long(e->m_qkv, d_lens, B, S, e->att_part, e->att_stats, e->ctx, st, H);
  };
  const void* final_h = e->h;
  const bool skinny = e->fused_ln && M <= skinny_max_tokens() && skinny_linear_supported(M, H, H, H) &&
                      skinny_linear_supported(M, 3 * H, H, H) && skinny_linear_supported(M, I, H, H) &&
                      skinny_linear_supported(M, H, I, H);
  if (skinny) {
    // A handful of tokens (batch-1 encode_query): the same deferred-LayerNorm dataflow as below, every linear layer
    // as a weight stream over all SMs (skinny_linear.cu); the row statistics are computed by the consumer itself.
    for (size_t l = 0; l < e->layers.size(); ++l) {
      LayerW* L = e->layers[l];
      const LayerW* P = l ? e->layers[l - 1] : nullptr;
      SkinnyArgs g{};
      g = SkinnyArgs{e->h, L->wqkv, L->bqkv, P ? L->cqkv : nullptr, nullptr, e->qkv, M, 3 * H, H, EPI_BIAS, P ? 1 : 0, eps, H};
      ICD_TRY(launch_skinny_linear(g, st));
      ICD_TRY(attention());
      g = SkinnyArgs{e->ctx, L->wo, L->bo_r, P ? P->ln2g : nullptr, e->h, e->t, M, H, H, EPI_BIAS_RESIDUAL, 0, eps, H};
      ICD_TRY(launch_skinny_linear(g, st));
      g = SkinnyArgs{e->t, L->w1, L->b1, L->c1, nullptr, e->f, M, I, H, EPI_BIAS_GELU, 1, eps, H};
      ICD_TRY(launch_skinny_linear(g, st));
      g = SkinnyArgs{e->f, L->w2, L->b2_r, L->ln1g, e->t, e->h, M, H, I, EPI_BIAS_RESIDUAL, 0, eps, H};
      ICD_TRY(launch_skinny_linear(g, st));
    }
    LayerW* L = e->layers.back();
    ICD_TRY(launch_layernorm(e->h, M, L->ln2g, L->ln2b, eps, e->h1, st, H));
    final_h = e->h1;
  } else if (e->fused_ln) {
    // Deferred LayerNorm: e->h carries the layer input -- normalised for layer 0 (embed_ln), the un-normalised
    // FFN-down output x2 = LN1(x1) + FFN(LN1(x1)) afterwards -- and e->t the un-normalised x1 = LN2(x2') + attn;
    // stats2 / stats1 hold their row statistics.  No LayerNorm launch until the one that closes the last layer.
    for (size_t l = 0; l < e->layers.size(); ++l) {
      LayerW* L = e->layers[l];
      const LayerW* P = l ? e->layers[l - 1] : nullptr;
      const bool last = l + 1 == e->layers.size();
      GemmArgs g{};
      g = GemmArgs{e->m_h, L->m_qkv, L->bqkv, nullptr, e->m_qkv_out, M, 3 * H, H, EPI_BIAS};
      if (P) g.vec2 = L->cqkv, g.stats_in = e->stats2;
      g.stats_stride = e->stats_stride, g.stats_cols = H, g.eps = eps;
      ICD_TRY(launch_gemm_tc(g, st));
      ICD_TRY(attention());
      // x1 = ctx Wo^T + bo + LN2'(x2')   (layer 0: + h)
      g = GemmArgs{e->m_ctx, L->m_o, L->bo_r, e->m_h, e->m_t, M, H, H, EPI_BIAS_RESIDUAL};
      if (P) g.vec2 = P->ln2g, g.stats_in = e->stats2;
      g.stats_out = e->stats1, g.stats_stride = e->stats_stride, g.stats_cols = H, g.eps = eps;
      ICD_TRY(launch_gemm_tc(g, st));
      // f = gelu(LN1(x1) W1^T + b1)
      g = GemmArgs{e->m_t, L->m_1, L->b1, nullptr, e->m_f, M, I, H, EPI_BIAS_GELU};
      g.vec2 = L->c1, g.stats_in = e->stats1, g.stats_stride = e->stats_stride, g.stats_cols = H, g.eps = eps;
      ICD_TRY(launch_gemm_tc(g, st));
      // x2 = f W2^T + b2 + LN1(x1)
      g = GemmArgs{e->m_f, L->m_2, L->b2_r, e->m_t, e->m_h, M, H, I, EPI_BIAS_RESIDUAL};
      g.vec2 = L->ln1g, g.stats_in = e->stats1, g.stats_stride = e->stats_stride, g.stats_cols = H, g.eps = eps;
      if (!last) g.stats_out = e->stats2;
      ICD_TRY(launch_gemm_tc(g, st));
    }
    LayerW* L = e->layers.back();
    ICD_TRY(launch_layernorm(e->h, M, L->ln2g, L->ln2b, eps, e->h1, st, H));
    final_h = e->h1;
  } else {
    for (size_t l = 0; l < e->layers.size(); ++l) {
      LayerW* L = e->layers[l];
      GemmArgs g{};
      // qkv = h Wqkv^T + b
      g = GemmArgs{e->m_h, L->m_qkv, L->bqkv, nullptr, e->m_qkv_out, M, 3 * H, H, EPI_BIAS};
      ICD_TRY(launch_gemm_tc(g, st));
      ICD_TRY(attention());
      // t = ctx Wo^T + bo + h ; h1 = LN(t)
      g = GemmArgs{e->m_ctx, L->m_o, L->bo, e->m_h, e->m_t, M, H, H, EPI_BIAS_RESIDUAL};
      ICD_TRY(launch_gemm_tc(g, st));
      ICD_TRY(launch_layernorm(e->t, M, L->ln1g, L->ln1b, eps, e->h1, st, H));
      // f = gelu(h1 W1^T + b1)
      g = GemmArgs{e->m_h1, L->m_1, L->b1, nullptr, e->m_f, M, I, H, EPI_BIAS_GELU};
      ICD_TRY(launch_gemm_tc(g, st));
      // t = f W2^T + b2 + h1 ; h = LN(t)
      g = GemmArgs{e->m_f, L->m_2, L->b2, e->m_h1, e->m_t, M, H, I, EPI_BIAS_RESIDUAL};
      ICD_TRY(launch_gemm_tc(g, st));
      ICD_TRY(launch_layernorm(e->t, M, L->ln2g, L->ln2b, eps, e->h, st, H));
    }
  }
  *final_h_out = final_h;
  *d_lens_out = d_lens;
  e->last_M = M;
  return ICD_OK;
}

}  // namespace icd

extern "C" {

int icd_encoder_forward(icd_encoder* e, const int32_t* ids, const int32_t* lens, int B, int S, void* out,
                        int out_dtype, void* stream, int sync) {
  ICD_CHECK_ARG(e != nullptr, "encoder is null");
  ICD_CHECK_ARG(B >= 0 && S >= 1 && S <= 512, "need 1 <= S <= 512");
  ICD_CHECK_ARG(S + e->pos_offset <= e->cfg.max_position, "S + position offset exceeds max_position");
  const int out_flags = out_dtype;
  out_dtype &= 0xff;
  ICD_CHECK_ARG(out_dtype == ICD_F32 || out_dtype == ICD_BF16, "unknown out dtype");
  if (B == 0) return ICD_OK;
  ICD_CHECK_ARG(ids && lens && out, "null buffer");
  ICD_CHECK_ARG((int64_t)B * S <= 0x7fffffffLL / 4, "batch too large");
  ICD_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int H = e->cfg.hidden;
  const bool host_out = !is_device_ptr(out);
  void* d_out = out;
  if (host_out) {
    const size_t need = (size_t)B * H * 4;
    if (need > e->out_cap) {
      if (e->out_stage) cudaFree(e->out_stage);
      e->out_stage = nullptr;
      e->out_cap = 0;
      ICD_CUDA(cudaMalloc(&e->out_stage, need));
      e->out_cap = need;
    }
    d_out = e->out_stage;
  }
  const void* final_h = nullptr;
  const int32_t* d_lens = nullptr;
  ICD_TRY(encode_hidden(e, ids, lens, B, S, st, &final_h, &d_lens));
  ICD_TRY(launch_pool_normalise(final_h, d_lens, B, S, d_out, out_flags, st, H));
  if (host_out) {
    ICD_CUDA(cudaMemcpyAsync(out, d_out, (size_t)B * H * (out_dtype == ICD_F32 ? 4 : 2), cudaMemcpyDeviceToHost, st));
  }
  // host inputs were handed to cudaMemcpyAsync above: pageable buffers are staged before that call returns, pinned
  // ones are read when the stream gets there -- with sync = 0 the caller keeps them untouched until then (the feeder
  // in engine/encoder.py double-buffers them behind events)
  if (sync || host_out) ICD_CUDA(cudaStreamSynchronize(st));
  return ICD_OK;
}

int icd_encoder_set_embedding_ids(icd_encoder* e, int32_t position_offset, int32_t unk_id) {
  ICD_CHECK_ARG(e != nullptr, "encoder is null");
  ICD_CHECK_ARG(position_offset >= 0 && position_offset < e->cfg.max_position, "position_offset outside [0, max_position)");
  ICD_CHECK_ARG(unk_id < e->cfg.vocab_size, "unk_id outside the vocabulary");
  e->pos_offset = position_offset;
  e->unk = unk_id < 0 ? default_unk(e->cfg) : unk_id;
  return ICD_OK;
}

int icd_encoder_set_token_head(icd_encoder* e, const float* weight, const float* bias, int labels) {
  ICD_CHECK_ARG(e != nullptr && weight != nullptr && bias != nullptr, "null argument");
  ICD_CHECK_ARG(labels >= 1 && labels <= ICD_MAX_LABELS, "labels must be in [1, ICD_MAX_LABELS]");
  ICD_CUDA(cudaSetDevice(e->device));
  const size_t wn = (size_t)labels * e->cfg.hidden;
  if (e->head_w) cudaFree(e->head_w);
  if (e->head_b) cudaFree(e->head_b);
  e->head_w = e->head_b = nullptr;
  e->head_labels = 0;
  ICD_CUDA(cudaMalloc((void**)&e->head_w, wn * 4));
  ICD_CUDA(cudaMalloc((void**)&e->head_b, (size_t)labels * 4));
  ICD_CUDA(cudaMemcpy(e->head_w, weight, wn * 4, cudaMemcpyDefault));
  ICD_CUDA(cudaMemcpy(e->head_b, bias, (size_t)labels * 4, cudaMemcpyDefault));
  e->head_labels = labels;
  return ICD_OK;
}

int icd_encoder_token_logits(icd_encoder* e, const int32_t* ids, const int32_t* lens, int B, int S, float* out,
                             void* stream, int sync) {
  ICD_CHECK_ARG(e != nullptr, "encoder is null");
  ICD_CHECK_ARG(e->head_labels > 0, "no token head: call icd_encoder_set_token_head first");
  ICD_CHECK_ARG(B >= 0 && S >= 1 && S <= 512, "need 1 <= S <= 512");
  ICD_CHECK_ARG(S + e->pos_offset <= e->cfg.max_position, "S + position offset exceeds max_position");
  if (B == 0) return ICD_OK;
  ICD_CHECK_ARG(ids && lens && out, "null buffer");
  ICD_CHECK_ARG((int64_t)B * S <= 0x7fffffffLL / 4, "batch too large");
  ICD_CUDA(cudaSetDevice(e->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int L = e->head_labels;
  const size_t bytes = (size_t)B * S * L * 4;
  const bool host_out = !is_device_ptr(out);
  float* d_out = out;
  if (host_out) {
    if (bytes > e->out_cap) {
      if (e->out_stage) cudaFree(e->out_stage);
      e->out_stage = nullptr;
      e->out_cap = 0;
      ICD_CUDA(cudaMalloc(&e->out_stage, bytes));
      e->out_cap = bytes;
    }
    d_out = (float*)e->out_stage;
  }
  const void* final_h = nullptr;
  const int32_t* d_lens = nullptr;
  ICD_TRY(encode_hidden(e, ids, lens, B, S, st, &final_h, &d_lens));
  ICD_TRY(launch_token_head(final_h, B * S, e->head_w, e->head_b, L, d_out, st, e->cfg.hidden));
  if (host_out) ICD_CUDA(cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, st));
  // host inputs were handed to cudaMemcpyAsync above: pageable buffers are staged before that call returns, pinned
  // ones are read when the stream gets there -- with sync = 0 the caller keeps them untouched until then (the feeder
  // in engine/encoder.py double-buffers them behind events)
  if (sync || host_out) ICD_CUDA(cudaStreamSynchronize(st));
  return ICD_OK;
}

int icd_encoder_read_hidden(icd_encoder* e, int reserved, float* out, int64_t count) {
  (void)reserved;
  ICD_CHECK_ARG(e && out, "null argument");
  ICD_CHECK_ARG(count == (int64_t)e->last_M * e->cfg.hidden, "count must be tokens*hidden of the last forward");
  ICD_CUDA(cudaSetDevice(e->device));
  float* tmp = nullptr;
  ICD_CUDA(cudaMalloc((void**)&tmp, (size_t)count * 4));
  int st = launch_bf16_to_f32(e->fused_ln ? e->h1 : e->h, tmp, count, 0);
  if (st == ICD_OK) {
    cudaError_t err = cudaMemcpy(out, tmp, (size_t)count * 4, cudaMemcpyDefault);
    if (err != cudaSuccess) {
      set_error("read_hidden: %s", cudaGetErrorString(err));
      st = ICD_E_CUDA;
    }
  }
  cudaFree(tmp);
  return st;
}

}  // extern "C"
