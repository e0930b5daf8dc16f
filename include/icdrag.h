/* icdrag.h -- C ABI of libicdrag.so, the B200 (sm_100a) engine behind the ICD-10 retrieval
 * hot path of yilane/rag-project-icd10.
 *
 * The reference has no FFI of its own: its hot path is two third-party Python objects,
 *   SentenceTransformer(...).encode        (services/embedding_service.py:61,81,97,120)
 *   MilvusClient(...).insert / .search     (services/milvus_service.py:259,280)
 * This header is what a binding for those two seams calls instead (ctypes stub in
 * INTEGRATION.md; the in-tree binding is rag-project-icd10_b200/_native.py).
 *
 * Conventions
 *   - every function returns an int status: 0 = ok, <0 = error (ICD_E_*); the message of the
 *     last error on the calling thread is icd_last_error().
 *   - the caller allocates every buffer; the library never frees caller memory. Handles are
 *     opaque and released by the matching *_destroy.
 *   - data pointers may be host or device pointers; the library classifies them with
 *     cudaPointerGetAttributes. Host inputs are copied in, host outputs copied back, inside
 *     the call (that is the "e2e" path bench.py times).
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream). With
 *     sync=0 and device OUTPUT buffers the call returns after enqueue (host INPUT buffers must
 *     then stay untouched until the stream has consumed them: pageable ones are staged before
 *     the call returns, pinned ones are read asynchronously); with host output buffers or
 *     sync=1 it returns when the results are in place.
 *   - one in-flight call per handle; distinct handles are independent.
 *   - there is NO CPU fallback: without a CUDA device every create call fails with
 *     ICD_E_CUDA.
 */
#ifndef ICDRAG_H_
#define ICDRAG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICD_OK 0
#define ICD_E_ARG (-1)      /* bad argument */
#define ICD_E_CUDA (-2)     /* CUDA runtime / driver error */
#define ICD_E_STATE (-3)    /* handle in the wrong state (e.g. encoder not finalised) */
#define ICD_E_NOMEM (-4)    /* device allocation failed */
#define ICD_E_UNSUPPORTED (-5)
#define ICD_E_NCCL (-6)

/* element types of vectors crossing the ABI */
#define ICD_F32 0
#define ICD_BF16 1
/* OR-ed into icd_encoder_forward's out_dtype: return the pooled mean without L2 normalisation
 * (SentenceTransformer.encode(normalize_embeddings=False)) */
#define ICD_OUT_NO_NORMALISE 0x100

/* level weighting of MilvusService.search (services/milvus_service.py:290-314,550-558) */
#define ICD_WEIGHT_RERANK 0 /* reference behaviour: raw top-k, then score*w(level), stable re-sort */
#define ICD_WEIGHT_PRE 1    /* weight every row before selection (NOT what the reference does) */
#define ICD_WEIGHT_NONE 2   /* raw inner product only */

/* scan kernel selection */
#define ICD_PATH_AUTO 0
#define ICD_PATH_STREAM 1 /* CUDA-core 128-bit HBM stream, exact fp32 accumulate (small batches) */
#define ICD_PATH_TENSOR 2 /* tcgen05/TMEM tensor-core scan with fused top-k epilogue */

/* index flags */
#define ICD_INDEX_KEEP_F32 1 /* keep an fp32 master copy of every row next to the bf16 table */

#define ICD_MAX_K 128
#define ICD_NCCL_ID_BYTES 128

typedef struct icd_index icd_index;
typedef struct icd_encoder icd_encoder;
typedef struct icd_shard_group icd_shard_group;

int icd_version(void);
const char* icd_last_error(void);
/* number of kernels this library has launched on the calling process so far (bench.py's gpu_launches) */
int64_t icd_launch_count(void);
int icd_device_count(void);
/* process-wide tuning knobs of the tensor-core scan (tests and profiling; defaults are right for
 * production): "scan_sample" (stride of the sampling pre-pass, 0 = off, -1 = by table size),
 * "scan_drift" (tiles a CTA may run ahead of its row group, 0 = off), "scan_tmax" (query tiles per
 * row stream per launch, default 16), "scan_kbs" /
 * "scan_kbs_pair" (K blocks per pipeline stage for single CTAs / CTA pairs, upper bounds: default 3 / 6),
 * "scan_pair" (CTA pairs: -1 auto, 0 off), "scan_qsplit" (last third of the query tile's K in shared
 * memory so that two accumulator buffers fit: -1 auto, 0 off), "scan_qtmem" (K blocks kept in TMEM when
 * split, 0 = all that fit), "scan_generic" (1 = the run-time-shaped MMA issue loop instead of the unrolled one), "scan_pre_slots"
 * (0 = the list-based sampling pre-pass instead of the slot-maxima one), "scan_small_pre" (0 = no pre-pass on tables
 * below 512 k rows), "enc_pdl" (0 = plain stream order between the
 * encoder's kernels instead of programmatic dependent launch), "enc_skinny" (forwards of few tokens -- batch-1
 * encode_query -- run their linear layers as a weight stream over all SMs instead of tile GEMMs: 1 = up to 64 tokens
 * (default), 0 = never; the two paths agree to bf16 rounding).
 * Results never depend on them.  Production builds read NO environment variables on the compute path; profiling
 * builds (-DICD_PROFILING) additionally honour ICD_SCAN_*, ICD_GEMM_PAIR, ICD_ENC_FUSED_LN, ICD_ATTN_DBG. */
int icd_tune(const char* key, int value);

/* ---------------------------------------------------------------- vector table + scan ------
 * Replaces the Milvus FLAT/IP collection: MilvusClient.insert (services/milvus_service.py:259)
 * and MilvusClient.search (services/milvus_service.py:280-285).  Rows are stored row-major
 * [n, dim] in bf16 (always) and optionally fp32 (ICD_INDEX_KEEP_F32); one level byte per row
 * (1,2,3; anything else weighs 1.0) feeds _calculate_level_weight (milvus_service.py:550-558).
 */
int icd_index_create(int dim, int device, int64_t capacity_rows, int flags, icd_index** out);
int icd_index_destroy(icd_index* idx);
/* append n rows; vecs is [n, dim] of `dtype`, level is [n] or NULL (all level 1).  Both
 * pointers live in the same memory space (host or device). Grows the table when needed. */
int icd_index_append(icd_index* idx, const void* vecs, int dtype, const uint8_t* level, int64_t n);
/* zero-copy: use caller-owned DEVICE buffers ([n, dim] bf16, [n] u8) as the table. The caller
 * keeps them alive; append/clear on an adopted index fail with ICD_E_STATE. */
int icd_index_adopt(icd_index* idx, const void* dev_bf16, const uint8_t* dev_level, int64_t n);
int icd_index_clear(icd_index* idx); /* drop_collection + re-create (milvus_service.py:359-367) */
int64_t icd_index_size(const icd_index* idx);
int icd_index_dim(const icd_index* idx);
/* copy rows [row0, row0+n) out as fp32 (from the master when kept, else widened bf16) */
int icd_index_read(const icd_index* idx, int64_t row0, int64_t n, float* out);

/* exact inner-product top-k of B queries against every row.
 *   q          [B, dim] of q_dtype (host or device)
 *   k          1..ICD_MAX_K; when the table holds fewer than k rows the tail is (-inf, -1)
 *   out_score  [B, k] level-weighted score (== out_raw for ICD_WEIGHT_NONE), may be NULL
 *   out_raw    [B, k] raw inner product, may be NULL
 *   out_id     [B, k] row ids (int64, + the shard's row offset when searched through a group)
 * Ordering: by (score desc, id asc) of the deciding score; ICD_WEIGHT_RERANK selects on the
 * raw score and then re-sorts the k hits by weighted score, ties keeping raw order -- the
 * reference's list.sort(key=score, reverse=True) (milvus_service.py:314). */
int icd_index_search(icd_index* idx, const void* q, int q_dtype, int B, int k, int weight_mode,
                     int path, float* out_score, float* out_raw, int64_t* out_id, void* stream,
                     int sync);
/* filtered search: the exact top-k over the rows a bitmap allows (a scalar `filter` expression evaluated on the host).
 *   row_mask   ceil(n/32) uint32 words, host or device (bit i&31 of word i>>5 = local row i may be returned); bits at or
 *              above n are ignored; NULL = all rows (== icd_index_search)
 *   mask_rows  must equal icd_index_size(idx), else ICD_E_ARG
 * Ordering, weight modes and the (-inf, -1) tail (fewer than k allowed rows) as icd_index_search.  A host mask is
 * copied into the handle's workspace like the queries. */
int icd_index_search_filtered(icd_index* idx, const void* q, int q_dtype, int B, int k, int weight_mode, int path,
                              const uint32_t* row_mask, int64_t mask_rows, float* out_score, float* out_raw,
                              int64_t* out_id, void* stream, int sync);
/* paged and range search beyond ICD_MAX_K (pymilvus's offset / limit and FLAT/IP range search).
 * Let L be the list icd_index_search_filtered would return with k = offset + limit if k could be that large: the same
 * canonical fp32 scores, (key desc, id asc) order, weight modes (ICD_WEIGHT_RERANK re-sorts the whole list of
 * offset + limit raw hits) and mask rules -- after the range flags have removed every row whose RAW inner product lies
 * outside (radius, range_filter] (Milvus's IP rule, in every weight mode).  The call writes L[offset, offset + limit)
 * as [B, limit]; slots past the end of L are (-inf, -1).
 *   page       offset >= 0, limit >= 1, offset + limit <= ICD_MAX_LIMIT; with both range flags radius < range_filter
 * row_mask / mask_rows as icd_index_search_filtered; buffers, stream and sync as icd_index_search.  Every workspace
 * size is known on the host, so the call enqueues without synchronising.  Exact by construction: every allowed row is
 * scored, then a radix select and a sort (DESIGN.md, "Paged search"); a [chunk, n] fp32 workspace (<= 512 MiB)
 * bounds the queries per pass. */
#define ICD_MAX_LIMIT 16384  /* offset + limit, as pymilvus */
#define ICD_RANGE_RADIUS 1   /* keep raw >  radius       */
#define ICD_RANGE_FILTER 2   /* keep raw <= range_filter */
typedef struct icd_search_page {
  int32_t offset, limit, range_flags;
  float radius, range_filter;
} icd_search_page;
int icd_index_search_page(icd_index* idx, const void* q, int q_dtype, int B, const icd_search_page* page,
                          int weight_mode, const uint32_t* row_mask, int64_t mask_rows, float* out_score,
                          float* out_raw, int64_t* out_id, void* stream, int sync);
/* kernels launched / microseconds of device time of the last search on this handle, split by
 * stage: [0] scan, [1] merge, [2] rescore+finalise.  For bench.py's roofline line. */
int icd_index_last_timing(const icd_index* idx, float* us3, int* launches);
int icd_index_set_timing(icd_index* idx, int enabled);   /* also restarts the call count below */
/* the same three stage times averaged over the searches issued since icd_index_set_timing(idx, 1)
 * (the most recent 64 of them); *calls = how many were averaged.  Synchronises with the last one only,
 * so a timed region of back-to-back searches is measured without host syncs in between. */
int icd_index_mean_timing(const icd_index* idx, float* us3, int* calls);
/* queries the tensor path could not certify exact and re-searched with the exact stream scan since the previous call
 * (waits for the device); the counter restarts at 0 */
int icd_index_take_fallbacks(icd_index* idx, int64_t* count);

/* ---------------------------------------------------------------- row-sharded scan ---------
 * New work (the reference is single-process): rank r holds rows [row_offset, row_offset+n_r);
 * every rank calls search with the same B queries; local top-k, exchange of k candidates per
 * query, merge; every rank gets the merged result. exchange: 0 = ncclAllGather, 1 = peer
 * stores over NVLink-mapped slabs (cudaIpc) written by the merge-prep kernel itself. */
int icd_nccl_unique_id(void* out128);
int icd_shard_group_create(const void* nccl_id128, int rank, int world, int64_t row_offset,
                           icd_index* local, icd_shard_group** out);
int icd_shard_group_destroy(icd_shard_group* g);
/* peer-slab wiring for exchange=1: each rank exports its slab handle (64 bytes), the caller
 * all-gathers them (any transport) and hands the table back. */
int icd_shard_group_export_slab(icd_shard_group* g, void* out_handle64);
int icd_shard_group_import_slabs(icd_shard_group* g, const void* handles /*[world][64]*/);
int icd_shard_group_search(icd_shard_group* g, const void* q, int q_dtype, int B, int k,
                           int weight_mode, int path, int exchange, float* out_score,
                           float* out_raw, int64_t* out_id, void* stream, int sync);
/* the same with a row mask over this rank's LOCAL rows (mask_rows == icd_index_size of the local table); every rank
 * passes the mask of its own rows, results carry global ids as above */
int icd_shard_group_search_filtered(icd_shard_group* g, const void* q, int q_dtype, int B, int k, int weight_mode,
                                    int path, int exchange, const uint32_t* row_mask, int64_t mask_rows,
                                    float* out_score, float* out_raw, int64_t* out_id, void* stream, int sync);

/* ---------------------------------------------------------------- encoder ------------------
 * Replaces the arithmetic of SentenceTransformer.encode(normalize_embeddings=True)
 * (services/embedding_service.py:81,97-102,120): BERT (post-LN, erf-GELU, learned absolute
 * positions) -> masked mean over tokens -> L2 normalise.  Tokenisation stays on the host.
 * XLM-RoBERTa encoders (the same layer, positions numbered from pad_token_id + 1) use the same
 * weight layout plus icd_encoder_set_embedding_ids.
 */
typedef struct icd_bert_cfg {
  int32_t vocab_size;   /* 21128 for text2vec-base-chinese */
  int32_t hidden;       /* 768 or 1024 */
  int32_t layers;       /* 12 */
  int32_t heads;        /* hidden / 64: 12 at 768, 16 at 1024 (head dim must be 64) */
  int32_t intermediate; /* 3072 */
  int32_t max_position; /* 512 */
  int32_t type_vocab;   /* 2 */
  float ln_eps;         /* 1e-12 */
} icd_bert_cfg;

/* number of fp32 values icd_encoder_create expects in `weights` for this config, in the
 * canonical order documented in rag-project-icd10_b200/engine/weights.py (HF BertModel names) */
int64_t icd_encoder_weight_count(const icd_bert_cfg* cfg);
int icd_encoder_create(const float* weights, int64_t count, const icd_bert_cfg* cfg, int device,
                       icd_encoder** out);
int icd_encoder_destroy(icd_encoder* enc);
/* Embedding conventions, read at each forward: token t of a sequence reads position row position_offset + t
 * (0 for BERT; pad_token_id + 1 = 2 for XLM-RoBERTa) and ids outside [0, vocab_size) read row unk_id (3 for
 * XLM-RoBERTa's <unk>).  Defaults: 0, and unk_id 100 ([UNK] of BERT vocabularies) when vocab_size > 100, else 0;
 * a negative unk_id restores that default.  S + position_offset must not exceed max_position. */
int icd_encoder_set_embedding_ids(icd_encoder* enc, int32_t position_offset, int32_t unk_id);
/* ids [B, S] int32 (0-padded), lens [B] int32 = number of real tokens (attention mask is
 * position < len); out [B, hidden] of out_dtype. S <= 512 (BERT's position table): S <= 128 -- the
 * sentence-transformers max_seq_length of text2vec-base-chinese -- is one tile of the tensor-core
 * attention kernel; longer sequences (the token-classification path) run the same kernel split over
 * 128-key tiles plus a combine pass. B*S <= the capacity given to icd_encoder_reserve. */
int icd_encoder_reserve(icd_encoder* enc, int max_tokens);
int icd_encoder_forward(icd_encoder* enc, const int32_t* ids, const int32_t* lens, int B, int S,
                        void* out, int out_dtype, void* stream, int sync);
/* parity hook: copy the LAST layer's hidden states (after its closing LayerNorm) of the last forward as fp32
 * [B*S, hidden] to a host/device buffer.  `reserved` must be 0 (intermediate layers are not kept: their streams are
 * overwritten in place). */
int icd_encoder_read_hidden(icd_encoder* enc, int reserved, float* out, int64_t count);

/* Token-classification head on the same encoder (SURVEY 8f rank 3): the per-token logits that
 * AutoModelForTokenClassification produces inside the reference's NER pipeline
 * (services/medical_ner_service.py:76-90, called at :182).  weight [labels, hidden] and bias [labels] are
 * classifier.weight / classifier.bias (fp32, host or device; copied).  labels <= ICD_MAX_LABELS. */
#define ICD_MAX_LABELS 64
int icd_encoder_set_token_head(icd_encoder* enc, const float* weight, const float* bias, int labels);
/* logits [B, S, labels] fp32 (host or device) for ids [B, S] / lens [B] as in icd_encoder_forward; positions
 * >= lens[b] hold the logits of padding tokens and are ignored by the caller, like the pipeline ignores them. */
int icd_encoder_token_logits(icd_encoder* enc, const int32_t* ids, const int32_t* lens, int B, int S,
                             float* out, void* stream, int sync);

/* ---------------------------------------------------------------- host tokeniser (encoder feeder) ------
 * Replaces the tokenisation step inside SentenceTransformer.encode (the model directory's BertTokenizerFast, reached
 * from services/embedding_service.py:81,97-102,120): BERT normaliser -> whitespace / punctuation split -> WordPiece
 * -> [CLS] ... [SEP], multi-threaded on the host, writing the int32 id rows icd_encoder_forward reads.
 *   tokens        the vocabulary, one token per line ('\n'-terminated UTF-8), n_tokens lines; ids[i] = id of line i
 *   char_class    [65536] per BMP code point: bits 0-1 kind (0 map, 1 whitespace, 2 remove, 3 fallback), bit 2 = CJK
 *                 ideograph (isolated), bit 3 = punctuation when it appears as an OUTPUT character
 *   map_offsets   [65537] / map_pool [pool_len]: normalised replacement code points of every kind-0 code point
 * (rag-project-icd10_b200/engine/tokenizer.py builds the tables from the Unicode database and decides which code
 * points are left to the wrapped reference tokenizer.) */
typedef struct icd_tokenizer icd_tokenizer;
int icd_tokenizer_create(const char* tokens, int64_t tokens_bytes, const int32_t* ids, int64_t n_tokens,
                         const uint8_t* char_class, const uint32_t* map_offsets, const uint32_t* map_pool,
                         int64_t pool_len, icd_tokenizer** out);
int icd_tokenizer_destroy(icd_tokenizer* tok);
/* texts: n UTF-8 strings joined by single NUL bytes (nbytes in total, no trailing NUL).  Row i of ids (row_stride
 * int32 per row, >= max_len) receives lens[i] ids including [CLS] / [SEP], truncated to max_len; entries past lens[i]
 * are left untouched.  needs_fallback[i] = 1 (and lens[i] = 0) when sentence i must go through the reference
 * tokenizer instead (fallback code point, supplementary plane, malformed UTF-8, literal special token).
 * threads <= 0: all hardware threads. */
int icd_tokenizer_encode(const icd_tokenizer* tok, const char* texts, int64_t nbytes, int64_t n, int max_len,
                         int32_t* ids, int row_stride, int32_t* lens, uint8_t* needs_fallback, int threads);
/* gather rows[b] (b < B) of such an id table into a zero-padded [B, S] batch + lens[B]: the ids / lens arguments of
 * icd_encoder_forward (host buffers; pinned ones make the H2D copy asynchronous) */
int icd_pack_batch(const int32_t* ids, int row_stride, const int32_t* lens, const int64_t* rows, int B, int S,
                   int32_t* out_ids, int32_t* out_lens);

#ifdef __cplusplus
}
#endif
#endif /* ICDRAG_H_ */
