/* marqo_b200 — C ABI of the B200-native embed-and-score engine.
 *
 * The reference (marqo-ai/marqo) has NO foreign-function interface on this path: it calls
 * open_clip / transformers / torch for the encoders and an HTTP POST to Vespa for the score
 * step.  This header is therefore the boundary a Marqo maintainer would bind from Python
 * (ctypes — see INTEGRATION.md) underneath the reference's two pure-Python seams:
 *
 *   B1  encoder seam   model.encode(...) objects held by s2_inference._available_models
 *                      (src/marqo/s2_inference/s2_inference.py:123-158, :520-568;
 *                       loaders map src/marqo/s2_inference/model_registry.py:2133-2145)
 *   B2  score seam     VespaClient.query()/feed_batch()
 *                      (src/marqo/vespa/vespa_client.py:198-242, :267-296), consumed at
 *                      src/marqo/tensor_search/tensor_search.py:2189 and
 *                      src/marqo/core/vespa_index/add_documents_handler.py:177
 *
 * Conventions: plain C, opaque handles, caller-owned host buffers, every function returns an
 * int status (B200_OK == 0) and leaves a thread-local message readable through
 * b200_last_error().  Handles are internally serialised (one mutex + one CUDA stream per
 * handle), so concurrent calls from Marqo's request threadpool are safe.  There is no CPU
 * fallback: without a usable sm_100 device every compute entry point fails with
 * B200_ERR_NO_DEVICE.
 */
#ifndef MARQO_B200_H
#define MARQO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_ABI_VERSION 1

enum b200_status {
    B200_OK = 0,
    B200_ERR_INVALID_ARG = 1,
    B200_ERR_NO_DEVICE = 2,
    B200_ERR_CUDA = 3,
    B200_ERR_OOM = 4,
    B200_ERR_UNSUPPORTED = 5,
    B200_ERR_INTERNAL = 6,
    B200_ERR_MISSING_WEIGHT = 7
};

int b200_abi_version(void);
/* Thread-local text of the last failure on this thread ("" if none). */
const char* b200_last_error(void);
/* Number of visible CUDA devices with compute capability 10.x. */
int b200_device_count(int* out_count);

/* Page-locked host memory (cudaHostAlloc, portable) for staging inputs: host-to-device copies from it run at the full
 * PCIe rate.  The reference stages every image separately (`.to(device)` per image at
 * src/marqo/tensor_search/add_docs.py:129-134); the adapters assemble a batch in one such buffer instead. */
int b200_host_alloc(size_t bytes, void** out);
int b200_host_free(void* p);

/* ===================================================================================== */
/* Score + top-k over a GPU-resident embedding matrix  (SURVEY §8 a8; replaces the Vespa   */
/* nearestNeighbor / closeness / top-k round trip specified by                            */
/* src/marqo/core/unstructured_vespa_index/unstructured_vespa_index.py:59-133,            */
/* src/marqo/core/structured_vespa_index/structured_vespa_index.py:403-446,645-688 and    */
/* src/marqo/core/unstructured_vespa_index/unstructured_vespa_schema.py:155-166,225-230). */
/* ===================================================================================== */

typedef struct b200_index b200_index;

/* Distance metrics: names from src/marqo/core/models/marqo_index.py:63-69. */
enum b200_metric {
    B200_METRIC_PRENORMALIZED_ANGULAR = 0, /* distance = 1 - q.e           closeness = 1/(1+d) */
    B200_METRIC_ANGULAR = 1,               /* distance = acos(cos(q,e))    closeness = 1/(1+d) */
    B200_METRIC_DOTPRODUCT = 2,            /* distance = -q.e              closeness = q.e (raw) */
    B200_METRIC_EUCLIDEAN = 3              /* distance = |q-e|             closeness = 1/(1+d)  (scan key 2 q.e - |e|^2) */
};

/* Create an empty row store of fp16[capacity_rows, dim] on `device` (grows on demand).
 * dim must be a multiple of 64 and <= 1024. */
int b200_index_create(int device, int dim, int metric, int64_t capacity_rows, b200_index** out);
int b200_index_destroy(b200_index* ix);

/* Append m chunk embeddings (fp32, host, row-major [m, dim]).  doc_ids[i] is the internal
 * document number (>= 0) the chunk belongs to; NULL means "one chunk per document, document
 * number == row number".  Rows of one document need not be contiguous.  Replaces
 * VespaClient.feed_batch for the tensor fields (vespa_client.py:267-296; the per-document
 * {"<chunk>": [floats]} blocks built at
 * src/marqo/core/semi_structured_vespa_index/semi_structured_document.py:127-143). */
int b200_index_add(b200_index* ix, const float* vecs, const int32_t* doc_ids, int64_t m);
/* Same, source already on the index's device (fp32 [m, dim]); used by the add_documents fast
 * path that never materialises List[List[float]] on the host. */
int b200_index_add_device(b200_index* ix, const float* d_vecs, const int32_t* d_doc_ids, int64_t m);
/* Same with the embeddings on the device (straight out of b200_model_encode_*_device) and the document numbers on the
 * host: the add_documents fast path — vectors never visit the host, the small id list does not need a device buffer
 * of the caller's (core/vespa_index/add_documents_handler.py:160-177 feeds what
 * core/inference/tensor_fields_container.py:196-223 collected). */
int b200_index_add_device_docs(b200_index* ix, const float* d_vecs, const int32_t* doc_ids, int64_t m);
/* Rows whose values are not finite or do not fit the fp16 row store (|x| > 65504 after the angular metric's
 * normalisation) are rejected by all three add calls with B200_ERR_INVALID_ARG; nothing of the batch is kept. */
/* Tombstone every row of a document (add_documents replaces by _id:
 * src/marqo/core/vespa_index/add_documents_handler.py:140,258).  O(rows): prefer b200_index_delete_rows when the
 * caller knows the document's rows. */
int b200_index_delete_doc(b200_index* ix, int32_t doc_id);
/* Tombstone the listed rows (the adapter keeps document -> rows): one small scatter per batch of replaced / deleted
 * documents instead of a corpus-wide pass per document. */
int b200_index_delete_rows(b200_index* ix, const int32_t* rows, int64_t n);
/* Squeeze tombstoned rows out of the matrix.  out_new_of_old: caller buffer of (current) num_rows int32 — the new row
 * number of every old row, -1 for a dead one; *out_rows = rows left.  Row numbers returned by earlier searches are
 * invalid afterwards. */
int b200_index_compact(b200_index* ix, int32_t* out_new_of_old, int64_t* out_rows);
int b200_index_num_rows(b200_index* ix, int64_t* out_rows);
int b200_index_info(b200_index* ix, int* out_dim, int* out_metric, int* out_device);
/* Copy row `row` back as fp32 (get_batch / use_existing_tensors:
 * add_documents_handler.py:160-165). */
int b200_index_get_row(b200_index* ix, int64_t row, float* out_vec);
int b200_index_get_rows(b200_index* ix, const int64_t* rows, int64_t n, float* out_vecs);

/* Exact search.  q: fp32 host [nq, dim].  For every query returns the k best DOCUMENTS under
 *   score(doc) = max over the document's live rows of closeness(q, row)
 * ordered by (score desc, doc_id asc).  out_doc/out_row/out_score are [nq, k]; unused slots are
 * filled with doc = row = -1, score = -inf.  out_row is the arg-max chunk row (Vespa's
 * closest(), used for _highlights: structured_vespa_index.py:942-1000).  out_score is the
 * closeness ("relevance", tensor_search.py:1771-1791) computed in fp64 from an exactly
 * rescored dot product. */
int b200_index_search(b200_index* ix, const float* q, int nq, int k, int32_t* out_doc, int32_t* out_row,
                      double* out_score);
/* How exactness is guaranteed (score.cu header): the tensor-core pass only SELECTS candidates, which are re-scored in
 * fp64; a per-query guard proves that no row outside the candidate set can reach the k-th exact score, and queries
 * that fail it (exact ties / near-ties across the candidate boundary, k beyond the per-SM lists) are answered by a
 * second threshold-collect pass over the corpus.  k <= 160 is normally ONE pass; any k <= 11000 is supported
 * (limit <= 1000 and offset <= 10000: src/marqo/api/configs.py:24-25). */
/* Same with queries and outputs resident on the index's device; asynchronous on the handle's
 * stream unless sync != 0.  With sync == 0 one fallback pass is enqueued unconditionally (it exits at once when no
 * query needs it); a query that would need MORE than one fallback pass cannot be driven from the host then —
 * b200_index_search_stats reports how often that happened (out_unresolved; 0 in every test and benchmark). */
int b200_index_search_device(b200_index* ix, const float* d_q, int nq, int k, int32_t* d_out_doc,
                             int32_t* d_out_row, double* d_out_score, int sync);
/* Counters since creation: groups of <= 64 queries searched, queries that failed the guard, fallback passes run by
 * the synchronous entry points, groups the asynchronous entry point left unresolved.  Any pointer may be NULL. */
int b200_index_search_stats(b200_index* ix, int64_t* out_groups, int64_t* out_flagged, int64_t* out_collect_passes,
                            int64_t* out_unresolved);

/* Search options: score modifiers (below) and a document FILTER.  filter_bits is a host bitset over LOCAL document
 * numbers (bit d of word d/32 set = document d may match; documents >= filter_docs are excluded): the adapter compiles
 * the ` AND <filter>` text Marqo appends to a tensor query (unstructured_vespa_index.py:59-66,135-226;
 * structured_vespa_index.py:690-793) to this bitset once per distinct filter string and the scan applies it where it
 * reads the row -> document map, next to the tombstone check — a filtered query costs one pass, whatever its
 * selectivity.  filter_tag != 0 names the bitset: the device copy is reused while tag and filter_docs repeat. */
typedef struct b200_search_opts {
    const int32_t* mult_cols;
    const double* mult_w;
    int32_t n_mult;
    const int32_t* add_cols;
    const double* add_w;
    int32_t n_add;
    const uint32_t* filter_bits;
    int64_t filter_docs;
    uint64_t filter_tag;
} b200_search_opts;
/* b200_index_search with options (opts == NULL: plain search). */
int b200_index_search_ex(b200_index* ix, const float* q, int nq, int k, const b200_search_opts* opts, int32_t* out_doc,
                         int32_t* out_row, double* out_score);

/* Score modifiers (SURVEY §8 f3).  Per-document numeric attributes: the `marqo__score_modifiers`
 * tensor<double>(p{}) field every document is fed with
 * (src/marqo/core/unstructured_vespa_index/unstructured_document.py:25,110-125;
 * src/marqo/core/semi_structured_vespa_index/semi_structured_document.py:23,104-117).  The host maps each
 * attribute NAME to a column number in [0, B200_MAX_ATTRIBUTE_COLUMNS).  values == NULL removes the cells (the
 * document no longer has the attribute); column == -1 with values == NULL removes the documents' cells in every
 * column (document overwritten or deleted).  Document numbers are LOCAL (before b200_index_set_doc_offset). */
#define B200_MAX_ATTRIBUTE_COLUMNS 64
int b200_index_set_attributes(b200_index* ix, int column, const int32_t* doc_ids, const double* values, int64_t n);
/* Many (column, document, value) cells in one call — one feed_batch, one launch. */
int b200_index_set_attributes_multi(b200_index* ix, const int32_t* columns, const int32_t* doc_ids, const double* values,
                                    int64_t n);
/* b200_index_search with the rank-profile function
 *   modify(score, mult_weights, add_weights) =
 *       if(count(mult_weights * attr) == 0, 1, reduce(mult_weights * attr, prod)) * score + reduce(add_weights * attr, sum)
 * (src/marqo/core/unstructured_vespa_index/unstructured_vespa_schema.py:266-271, applied at :225-230) evaluated
 * inside the scan, before top-k; `score` = closeness of the document's best chunk.  The sparse products run over the
 * attribute cells a document has.  mult_cols/mult_w and add_cols/add_w are the query tensors
 * `marqo__mult_weights_tensor` / `marqo__add_weights_tensor` (src/marqo/core/vespa_index/vespa_index.py:124-150;
 * src/marqo/core/constants.py:22-27) as (column, weight) lists, at most 16 each, evaluated in list order in fp64.
 * out_score is the MODIFIED score; order (score desc, doc asc).  B200_ERR_UNSUPPORTED when some document's
 * multiplier is negative on an index with explicit document ids (best chunk != best modified chunk). */
int b200_index_search_modified(b200_index* ix, const float* q, int nq, int k, const int32_t* mult_cols,
                               const double* mult_w, int n_mult, const int32_t* add_cols, const double* add_w, int n_add,
                               int32_t* out_doc, int32_t* out_row, double* out_score);

/* use_external != 0: run this handle's work on the caller's CUDA stream (a cudaStream_t, e.g. torch's current
 * stream; the value 0 is the legacy default stream).  use_external == 0 restores the handle's private stream. */
int b200_index_set_stream(b200_index* ix, void* cuda_stream, int use_external);
/* Device time (ms, CUDA events on the handle's stream) of the scan / merge kernels of the last
 * search call; used by bench.py for the roofline numerator. */
int b200_index_last_timing(b200_index* ix, float* scan_ms, float* merge_ms);
/* Row-sharded corpora: every document number returned by this index is offset by `offset` (the global number of
 * the shard's document 0), so per-shard results can be all-gathered and merged without a fix-up pass. */
int b200_index_set_doc_offset(b200_index* ix, int32_t offset);
/* Device-side merge of all-gathered per-shard results.  d_gathered holds, per shard, the packed block
 * {int32 doc[nq,k] | int32 row[nq,k] | double score[nq,k]} (what b200_index_search_device writes when its three
 * outputs point into one 16*nq*k-byte buffer); blocks are nq*k*16 bytes apart.  nshards*k <= 256. */
int b200_topk_merge_device(b200_index* ix, const void* d_gathered, int nshards, int nq, int k, int32_t* d_out_doc,
                           int32_t* d_out_row, double* d_out_score, int sync);
/* Fused exchange + merge over NVLink peer memory (SURVEY §8e "peer-stores into a symmetric buffer in the top-k
 * epilogue"): one process per GPU; every rank creates an exchange buffer, the ranks swap the 64-byte handles through
 * whatever transport they have (torch.distributed all_gather of a byte tensor), open each other's buffers, and then
 * b200_index_search_exchange = local search + ONE kernel that stores the packed [nq, k] block into every peer's
 * buffer, publishes it with a release flag, waits for the peers' blocks and merges them — no NCCL call on the query
 * path.  All ranks must call it the same number of times with the same nq and k (nq <= 64, world * k <= 256). */
typedef struct b200_exchange b200_exchange;
#define B200_EXCHANGE_HANDLE_BYTES 64
int b200_exchange_create(int device, int rank, int world, int max_nq, int max_k, b200_exchange** out,
                         void* out_handle /* B200_EXCHANGE_HANDLE_BYTES */);
/* handles: world * B200_EXCHANGE_HANDLE_BYTES bytes, rank order (this rank's own entry is ignored). */
int b200_exchange_open(b200_exchange* ex, const void* handles);
int b200_exchange_destroy(b200_exchange* ex);
/* d_local_block: device scratch of nq * k * 16 bytes (this rank's packed block); outputs [nq, k] on the device. */
int b200_index_search_exchange(b200_index* ix, b200_exchange* ex, const float* d_q, int nq, int k, void* d_local_block,
                               int32_t* d_out_doc, int32_t* d_out_row, double* d_out_score, int sync);
/* Merge `nshards` per-shard result lists ([nshards, nq, k] each, host) into the global top-k
 * with the same total order; doc ids must already be global.  Used after the NCCL all-gather
 * of per-shard lists. */
int b200_topk_merge(int nshards, int nq, int k, const int32_t* doc, const int32_t* row, const double* score,
                    int32_t* out_doc, int32_t* out_row, double* out_score);
/* Binary snapshot of the row store (persistence / restart). */
int b200_index_save(b200_index* ix, const char* path);
int b200_index_load(int device, const char* path, b200_index** out);

/* ===================================================================================== */
/* Encoders (SURVEY §8 a2-a5): CLIP ViT image tower, CLIP text tower, BERT (e5).          */
/* Replace model.encode_image / encode_text / AutoModel forward called at                 */
/* src/marqo/core/inference/embedding_models/open_clip_model.py:249-286 and               */
/* src/marqo/core/inference/embedding_models/hugging_face_model.py:172-214.               */
/* ===================================================================================== */

typedef struct b200_model b200_model;

enum b200_arch {
    B200_ARCH_CLIP = 0, /* open_clip CLIP: vision tower + text tower */
    B200_ARCH_BERT = 1, /* HF BertModel + pooling */
    B200_ARCH_MPNET = 2 /* HF MPNetModel + pooling (all-mpnet-base-v2 family): post-LN blocks as BERT with LayerNorm eps
                           1e-5, a learned relative-position bias in every attention, no token-type embedding, position
                           ids from 2 (padding index 1); text.ctx = max_position_embeddings (514), so sequences are at
                           most ctx - 2 tokens; type_vocab is ignored */
};
enum b200_act { B200_ACT_GELU = 0, B200_ACT_QUICKGELU = 1 };
enum b200_pool { B200_POOL_MEAN = 0, B200_POOL_CLS = 1 };

typedef struct b200_tower_desc {
    int32_t width;      /* hidden size */
    int32_t layers;     /* transformer blocks */
    int32_t heads;      /* head_dim = width / heads must be 64 */
    int32_t mlp;        /* MLP hidden size */
    int32_t ctx;        /* text: context length (77 / 512); vision: unused */
    int32_t vocab;      /* text: vocabulary size; vision: unused */
    int32_t image_size; /* vision: 224 */
    int32_t patch;      /* vision: 32 / 14 */
} b200_tower_desc;

typedef struct b200_model_desc {
    int32_t arch;      /* enum b200_arch */
    int32_t embed_dim; /* output dimension (CLIP projection dim; BERT / MPNet: == width) */
    int32_t act;       /* enum b200_act */
    int32_t pool;      /* BERT / MPNet: enum b200_pool (hugging_face_model.py:205-214) */
    int32_t type_vocab; /* BERT only: token_type vocabulary (2) */
    int32_t max_batch; /* workspace sizing: largest number of items per encode call */
    float image_mean[3]; /* Normalize() constants, src/marqo/s2_inference/clip_utils.py:32-33 */
    float image_std[3];
    b200_tower_desc vision; /* CLIP only */
    b200_tower_desc text;   /* CLIP text tower, or the BERT / MPNet encoder */
} b200_model_desc;

int b200_model_create(int device, const b200_model_desc* desc, b200_model** out);
int b200_model_destroy(b200_model* m);
/* Upload one parameter (fp32, host, contiguous) under its checkpoint name: open_clip
 * state_dict names for CLIP ("visual.conv1.weight", "transformer.resblocks.0.attn.in_proj_weight",
 * ...), HF BertModel names for BERT ("embeddings.word_embeddings.weight", ...), HF MPNetModel names for MPNet
 * ("encoder.layer.0.attention.attn.q.weight", "encoder.relative_attention_bias.weight" [32, heads], ...). */
int b200_model_load_tensor(b200_model* m, const char* name, const float* data, int64_t numel);
/* Verifies every required parameter has been supplied, builds derived buffers. */
int b200_model_finalize(b200_model* m);

/* Images as uint8 HWC (host), all n of size h x w: resize (bicubic, shortest side) ->
 * centre-crop -> /255 -> Normalize -> ViT -> proj -> optional L2 normalise.
 * Replaces preprocessors['image'](pil).to(device) (src/marqo/tensor_search/add_docs.py:129-134)
 * + OPEN_CLIP.encode_image (open_clip_model.py:249-266).  out: fp32 host [n, embed_dim].
 * The /255 and Normalize steps happen inside the patch-embedding GEMM's operand load (its gather warps read the uint8
 * pixels and write bf16 into the tensor core's shared-memory operand): no normalised image or patch matrix exists in HBM
 * (SURVEY §8 a2; images already of the model's size skip the resize pass as well). */
int b200_model_encode_images_u8(b200_model* m, const uint8_t* hwc, int n, int h, int w, int normalize,
                                float* out);
/* Already-preprocessed fp32 CHW tensors [n,3,S,S] (the reference passes these through
 * unchanged: abstract_clip_model.py:108-111). */
int b200_model_encode_images_f32(b200_model* m, const float* chw, int n, int normalize, float* out);
/* Token ids int32 [n, seq] (host).  CLIP: causal text tower, EOT = arg-max id pooling.
 * BERT: attn_mask int32 [n, seq] (1 = token, 0 = pad; NULL = all ones), token_type 0.
 * MPNet: as BERT; token t of a row has position id 2 + t, pad tokens (mask 0) position id 1. */
int b200_model_encode_tokens(b200_model* m, const int32_t* ids, const int32_t* attn_mask, int n, int seq,
                             int normalize, float* out);
/* Device-resident variants: inputs/outputs are device pointers on the model's device,
 * asynchronous on the model's stream unless sync != 0. */
int b200_model_encode_images_u8_device(b200_model* m, const uint8_t* d_hwc, int n, int h, int w, int normalize,
                                       float* d_out, int sync);
int b200_model_encode_tokens_device(b200_model* m, const int32_t* d_ids, const int32_t* d_attn_mask, int n,
                                    int seq, int normalize, float* d_out, int sync);
int b200_model_set_stream(b200_model* m, void* cuda_stream, int use_external);
/* Optional per-kernel-class device timing: when enabled every GEMM / attention launch of an encode call is
 * bracketed by CUDA events on the handle's stream; b200_model_profile returns their sums over every encode call
 * since profiling was last (re-)enabled. */
int b200_model_set_profiling(b200_model* m, int enable);
int b200_model_profile(b200_model* m, float* gemm_ms, int* gemm_launches, float* attention_ms, int* attention_launches);
/* Device time (ms) of the last encode call and the number of kernels it launched. */
int b200_model_last_timing(b200_model* m, float* ms, int* launches);

/* Weighted-mean fusion + renormalise on the host-side contract of
 * src/marqo/tensor_search/tensor_search.py:1953-1973 and
 * src/marqo/core/inference/tensor_fields_container.py:355-365:
 * out = mean_i(w_i * v_i); if normalize and |out| > 0: out /= |out|.  fp64 arithmetic. */
int b200_fuse_vectors(const double* vecs, const double* weights, int n, int dim, int normalize, double* out);

/* ===================================================================================== */
/* Tokenizers (SURVEY §8 f2): text -> int32 token ids on the host, multi-threaded.       */
/* ===================================================================================== */

typedef struct b200_tokenizer b200_tokenizer;

/* WordPiece — what AutoTokenizer.from_pretrained(<BERT / e5 checkpoint>) gives the reference
 * (src/marqo/core/inference/embedding_models/hugging_face_model.py:125-130) and what encode() calls as
 * tokenizer(sentences, padding=True, truncation=True, max_length=...) (:179-185).  vocab_utf8: the bytes of vocab.txt
 * (one token per line, id = line number; must contain [PAD] [UNK] [CLS] [SEP]).  do_lower_case != 0 also strips
 * accents (BertNormalizer's strip_accents=None follows lowercase). */
int b200_tokenizer_create_wordpiece(const char* vocab_utf8, size_t nbytes, int do_lower_case, b200_tokenizer** out);
/* The same WordPiece with other special tokens: cls / sep frame every row, pad fills it, unk replaces unknown words;
 * all four must be in the vocabulary.  MPNet's tokenizer is ("<s>", "</s>", "<pad>", "[UNK]").  Together with the four,
 * the mask token is matched verbatim in the text when it is in the vocabulary: "[MASK]" when cls is "[CLS]", "<mask>"
 * otherwise.  b200_tokenizer_create_wordpiece is this call with ("[CLS]", "[SEP]", "[PAD]", "[UNK]"). */
int b200_tokenizer_create_wordpiece_special(const char* vocab_utf8, size_t nbytes, int do_lower_case, const char* cls,
                                            const char* sep, const char* pad, const char* unk, b200_tokenizer** out);
/* CLIP byte-level BPE — open_clip's SimpleTokenizer, the tokenizer OPEN_CLIP.load_tokenizer() returns for non-hf-hub
 * models (src/marqo/core/inference/embedding_models/open_clip_model.py:211-222; cleaning rules restated at
 * src/marqo/core/inference/embedding_models/hf_tokenizer.py:9-17).  merges_utf8: the DECOMPRESSED bytes of
 * bpe_simple_vocab_16e6.txt (line 1 is a header; at most 49152-256-2 merges are used).  ftfy.fix_text is not
 * restated: text that ftfy would repair (mojibake) tokenises as written. */
int b200_tokenizer_create_clip_bpe(const char* merges_utf8, size_t nbytes, b200_tokenizer** out);
int b200_tokenizer_destroy(b200_tokenizer* t);
int b200_tokenizer_vocab_size(b200_tokenizer* t, int* out_size);
/* Encode n UTF-8 strings (texts[i], text_bytes[i] bytes; invalid sequences decode as U+FFFD).
 * WordPiece: "[CLS] ids [SEP]", truncated to max_length, every row padded with [PAD] to the LONGEST row of this call
 * (padding=True): *out_seq_len = that length <= max_length.  CLIP BPE: "<start_of_text> ids <end_of_text>", truncated
 * to max_length (= context_length) with the last id forced to <end_of_text>, zero padded: *out_seq_len = max_length.
 * out_ids / out_mask (mask may be NULL): caller buffers of n * max_length int32; rows are written back to back with
 * stride *out_seq_len.  max_length >= 2.  Thread-safe (the handle is immutable after creation). */
int b200_tokenizer_encode(b200_tokenizer* t, const char* const* texts, const int64_t* text_bytes, int n, int max_length,
                          int32_t* out_ids, int32_t* out_mask, int* out_seq_len);

/* Recommender interpolation (SURVEY §8 f3): src/marqo/core/utils/vector_interpolation.py —
 * Lerp.interpolate :49-88 (sum_i (w_i / sum w) v_i), Nlerp.interpolate :91-119 (Lerp, then / |.|),
 * Slerp hierarchical :121-193,211-237.  vecs: fp64 [n, dim] host; out: fp64 [dim].  Host-side fp64 arithmetic in
 * the reference's order (these are <= a few dozen vectors per recommend call, src/marqo/core/search/recommender.py:88).
 * On the reference's error conditions returns B200_ERR_INVALID_ARG and stores which one in *out_error_kind so the
 * binding can raise ZeroSumWeightsError / ZeroMagnitudeVectorError / ValueError like the reference. */
enum b200_interp_method { B200_INTERP_LERP = 0, B200_INTERP_NLERP = 1, B200_INTERP_SLERP = 2 };
enum b200_interp_error {
    B200_INTERP_OK = 0,
    B200_INTERP_ZERO_SUM_WEIGHTS = 1, /* ZeroSumWeightsError      (:12, :74-77, :226-228) */
    B200_INTERP_ZERO_MAGNITUDE = 2,   /* ZeroMagnitudeVectorError (:16, :113-116) */
    B200_INTERP_ZERO_LENGTH = 3       /* ValueError               (:171-173) */
};
int b200_interpolate_vectors(const double* vecs, const double* weights, int n, int dim, int method, double* out,
                             int* out_error_kind);

/* ===================================================================================== */
/* Image decode (SURVEY §8 f4): baseline JPEG -> uint8 HWC RGB on the GPU.               */
/* Replaces the Pillow decode on Marqo's download threads (Image.open at                  */
/* src/marqo/core/inference/image_download.py:146-152, pixels materialised by the         */
/* transform at src/marqo/tensor_search/add_docs.py:129-134).  Huffman decoding runs on   */
/* the host (images of a batch in parallel); dequantisation + integer IDCT, fancy chroma  */
/* upsampling and YCbCr -> RGB run in two CUDA kernels over the whole batch and reproduce */
/* libjpeg-turbo's default decode (what Pillow returns) bit for bit.                      */
/* ===================================================================================== */

/* Size of a JPEG and whether this decoder handles it (baseline / extended-sequential Huffman, 8-bit, grey or YCbCr
 * with 4:4:4 / 4:2:2 / 4:2:0 sampling).  *out_supported == 0: decode it with Pillow (b200_last_error says why). */
int b200_jpeg_info(const uint8_t* file, size_t nbytes, int32_t* out_height, int32_t* out_width, int32_t* out_supported);
/* Decode n files.  d_out[i]: device buffer of heights[i] * widths[i] * 3 bytes on `device` (sizes from b200_jpeg_info, or
 * from a first call with d_out[i] == NULL, which only fills heights / widths / status).  status[i]: B200_OK,
 * B200_ERR_UNSUPPORTED (fall back to Pillow for this image) or B200_ERR_INVALID_ARG (no output buffer).  Synchronous. */
int b200_jpeg_decode_batch(int device, const uint8_t* const* files, const size_t* nbytes, int n, uint8_t* const* d_out,
                           int32_t* heights, int32_t* widths, int32_t* status);

/* ===================================================================================== */
/* Diagnostics: run ONE kernel of the encoder on host data (used by the kernel-level     */
/* numerics tests; not part of the reference-facing surface).                            */
/* ===================================================================================== */

/* out[M,N] = act(A[M,K] @ W[N,K]^T + bias) (+ residual); A and W are rounded to bf16 on the device, fp32
 * accumulate; act: 0 none, 1 erf-GELU, 2 QuickGELU; bias/residual may be NULL; out_bf16 != 0 rounds the result to
 * bf16 before it is returned as fp32.  in_place != 0 (needs a residual and fp32 output): the device output buffer IS
 * the residual buffer, as in the model's out_proj / fc2, which add onto the residual stream they overwrite. */
int b200_debug_gemm(int device, const float* A, const float* W, const float* bias, const float* residual, int M, int N,
                    int K, int act, int out_bf16, int in_place, float* out);
/* ViT patch embedding of uint8 HWC images [n,S,S,3]: ToTensor + Normalize (mean3/std3) -> conv1 (conv_w fp32
 * [N, 3*patch*patch], no bias) -> token rows: out fp32 [n*(G+1), N], row b*(G+1)+1+i = patch i of image b (+ pos[1+i]
 * when pos != NULL), class-token rows left zero.  use_gather != 0: the fused gather GEMM (no patch matrix in HBM,
 * src/marqo/tensor_search/add_docs.py:129-134 folded into the operand load); 0: im2col kernel + plain GEMM. */
int b200_debug_patch_embed(int device, const uint8_t* hwc, int n, int S, int patch, const float* conv_w, int N,
                           const float* mean3, const float* std3, const float* pos, int use_gather, float* out);
/* softmax(q k^T / 8 + mask) v over packed qkv fp32 [B*S, 3*W] (rounded to bf16); mask: 0 none, 1 causal,
 * 2 key length (kv_len int32 [B]).  out fp32 [B*S, W]. */
int b200_debug_attention(int device, const float* qkv, int B, int S, int W, int H, int mask, const int32_t* kv_len,
                         float* out);
/* b200_debug_attention with MPNet's relative-position bias: score(i, j) += rel_bias[bucket(j - i)][h] (rel_bias fp32
 * [32, H], host; bucket as transformers' MPNetEncoder.relative_position_bucket).  mask: 0 none or 2 key length. */
int b200_debug_attention_relbias(int device, const float* qkv, int B, int S, int W, int H, int mask,
                                 const int32_t* kv_len, const float* rel_bias, float* out);
/* The library's relative-position buckets (host only, no device): out[d + max_distance] = bucket(d) for
 * d = key - query in [-max_distance, max_distance]. */
int b200_debug_relative_position_buckets(int max_distance, int32_t* out);
/* LayerNorm over rows of fp32 [rows, w]. */
/* Mean device time (ms, CUDA events) of `iters` back-to-back attention launches on device-generated data. */
int b200_debug_attention_time(int device, int B, int S, int W, int H, int mask, int iters, float* out_ms);
int b200_debug_layernorm(int device, const float* x, const float* gamma, const float* beta, float eps, int rows, int w,
                         float* out);
/* The JPEG decoder's arithmetic (shared __host__ __device__ code of the two kernels) run on the host: lets the CPU test
 * suite pin it against Pillow pixel for pixel.  A test hook, not a product path.  out_rgb == NULL: size query. */
int b200_debug_jpeg_decode_host(const uint8_t* file, size_t nbytes, uint8_t* out_rgb, size_t out_capacity,
                                int32_t* out_height, int32_t* out_width);
/* Pillow-compatible bicubic resize (shortest side -> S) + centre crop of uint8 HWC images [n,h,w,3] -> [n,S,S,3]. */
int b200_debug_resize(int device, const uint8_t* hwc, int n, int h, int w, int S, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif /* MARQO_B200_H */
