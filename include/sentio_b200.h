/*
 * sentio_b200.h -- C ABI of libsentio_b200.so: the B200-native retrieve -> fuse -> rerank hot path.
 *
 * The reference (chernistry/sentio @ 68a63b1b) has no FFI: its "plugin API" is Python duck typing
 * (`retriever.retrieve(query, top_k)` src/core/graph/nodes.py:70, `reranker.rerank(query=, docs=, top_k=)`
 * src/core/graph/nodes.py:179-183).  Every entry point below therefore cites the reference *function* whose
 * arithmetic it replaces; the Python classes in sentio_b200/ keep the reference's names/signatures and call
 * these through ctypes (see INTEGRATION.md for the reference-side stub).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.
 *   - every function returns 0 on success, <0 on failure; sb_last_error() returns a thread-local message.
 *   - functions WITHOUT a `_dev` suffix take HOST buffers; host<->device copies happen inside the call on the
 *     context's stream and the call returns after the results are on the host.
 *   - functions WITH a `_dev` suffix take DEVICE buffers (e.g. torch tensor data_ptr()) and a cudaStream_t
 *     passed as void* (NULL = the context's own stream); they only enqueue work.
 *   - a context may be used from several host threads (the reference dispatches retrieve_async to a thread pool,
 *     src/core/retrievers/base.py:37-42); calls on one context are serialised by an internal mutex.
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef SENTIO_B200_H
#define SENTIO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sb_ctx sb_ctx;

/* status codes */
#define SB_OK 0
#define SB_ERR_CUDA (-1)
#define SB_ERR_ARG (-2)
#define SB_ERR_STATE (-3)
#define SB_ERR_UNSUPPORTED (-4)

/* dtypes accepted by sb_dense_load */
#define SB_F32 0
#define SB_F16 1

/* BM25 variants (rank_bm25 0.2.2 class names; reference src/core/retrievers/sparse.py:91-97) */
#define SB_BM25_OKAPI 0
#define SB_BM25_PLUS 1

/* fusion methods (reference src/core/retrievers/hybrid.py:223-259) */
#define SB_FUSE_RRF 0
#define SB_FUSE_WEIGHTED_RRF 1
#define SB_FUSE_COMB_SUM 2

/* ---------------------------------------------------------------- context ---------------------------------- */
int sb_create(int device, sb_ctx** out);
void sb_destroy(sb_ctx* ctx);
const char* sb_last_error(void);
/* library/ABI version (major*1000+minor) and number of SMs of the context's device */
int sb_version(void);
int sb_num_sms(sb_ctx* ctx);
/* blocks until everything enqueued on the context's stream has finished */
int sb_sync(sb_ctx* ctx);
/* the context's cudaStream_t (as void*), so torch can order its own work against it */
void* sb_stream(sb_ctx* ctx);
/*
 * Page-locked host buffers for callers that reuse their I/O arrays (a server's request / response rings): the host
 * entry points below detect page-locked pointers (cudaPointerGetAttributes) and then copy straight between the
 * caller's buffer and the device -- no staging memcpy on either side.  Pageable pointers work as before (staged).
 */
void* sb_host_alloc(size_t bytes);
void sb_host_free(void* p);
/* number of kernels this library has launched on behalf of the context (bench.py's gpu_launches) */
int64_t sb_launch_count(sb_ctx* ctx);
/*
 * Optional per-kernel timing for the roofline leg of bench.py: when enabled every launch of the kernels below is
 * bracketed by a CUDA event pair on the launching stream; sb_profile_read drains the finished pairs of one kernel id
 * (0 dense_scan, 1 dense_merge, 2 bm25_score, 3 bm25_select+final, 4 fuse, 5 cross-encoder forward, 6 dense sampling
 * passes + threshold select) and returns the
 * launch count and the summed device time in milliseconds.
 */
int sb_profile(sb_ctx* ctx, int enable);
int sb_profile_read(sb_ctx* ctx, int kernel_id, int64_t* n_out, double* ms_out);

/* ---------------------------------------------------------------- K1: dense cosine top-k -------------------- */
/*
 * Replaces the Qdrant `client.search(collection, query_vector, limit=top_k)` call behind
 * DenseRetriever.retrieve (reference src/core/retrievers/dense.py:41-64; collection created with
 * distance="Cosine", src/core/vector_store/qdrant_store.py:51-52).
 *
 * sb_dense_load: copies `n` row-major vectors of dimension `d` (host memory, dtype SB_F32 or SB_F16) into HBM as
 * fp16 rows (+ one fp32 inverse norm per row).  SB_F32 input is L2-normalised then rounded to fp16 (Qdrant's
 * "normalise at upsert"); SB_F16 input is stored verbatim.  The cosine is always evaluated exactly (fp64) against
 * the STORED fp16 values.  Doc i gets id `id_base + i` (shard-local -> global id).  Nothing is retained on the host.
 * `slot` selects one of SB_MAX_DENSE_SLOTS independent indexes (slot 1 = the reference's optional "web_cache"
 * collection, hybrid.py:146-182).
 */
#define SB_MAX_DENSE_SLOTS 2
int sb_dense_load(sb_ctx* ctx, int slot, const void* vecs, int64_t n, int32_t d, int32_t dtype, int64_t id_base);
/*
 * Scan selection: 0 = auto (batches of >= 16 queries use the tcgen05 batched-query scan, smaller ones the CUDA-core
 * scan), 1 = CUDA-core scan only; any other mode is SB_ERR_ARG.  Results are identical in both modes.
 */
int sb_dense_set_mode(sb_ctx* ctx, int mode);
int64_t sb_dense_count(sb_ctx* ctx, int slot);
int32_t sb_dense_dim(sb_ctx* ctx, int slot);
/*
 * sb_dense_topk: B queries (row-major B x d fp32, need not be normalised: any scale), best-first top-k per query, k <= 1024:
 * out_ids[B*k], out_scores[B*k] (exact fp64 cosine, ties broken by ascending id), out_counts[B] (= min(k, n)).
 * The result is the EXACT top-k of the stored rows for every input: the scans rank by an approximate cosine with a per-query
 * error bound eps, every row within 2 eps of the k-th best approximate score is re-scored in fp64, and a query whose window
 * cannot be served that way is answered by a brute-force fp64 kernel (DESIGN.md K1 "Exactness").  Page-locked q / out_*
 * buffers (sb_host_alloc) are used in place, pageable ones are staged.
 */
int sb_dense_topk(sb_ctx* ctx, int slot, const float* q, int32_t B, int32_t k,
                  int64_t* out_ids, double* out_scores, int32_t* out_counts);
int sb_dense_topk_dev(sb_ctx* ctx, int slot, const float* q_dev, int32_t B, int32_t k,
                      int64_t* out_ids_dev, double* out_scores_dev, int32_t* out_counts_dev, void* stream);
/* copies stored (fp16 -> fp32) rows of the given ids back to the host: out[n_ids * d]; used by tests/tools */
int sb_dense_fetch(sb_ctx* ctx, int slot, const int64_t* ids, int32_t n_ids, float* out);

/* ---------------------------------------------------------------- K2: BM25 ---------------------------------- */
/*
 * Replaces rank_bm25 0.2.2 BM25Okapi/BM25Plus.get_scores + np.argsort top-k + `score > 0` filter
 * (reference call sites src/core/retrievers/sparse.py:177-198).
 *
 * sb_bm25_load: term-major CSR postings.  indptr[V+1] (int64), post_doc[nnz] (int32 shard-local doc index,
 * ascending inside each term), post_tf[nnz] (uint16 term frequency), doc_len[n_docs] (int32), corpus-global
 * avgdl and idf[V] (fp64, already epsilon-floored for Okapi), variant, k1, b, delta.  Doc i gets id id_base + i.
 */
int sb_bm25_load(sb_ctx* ctx, const int64_t* indptr, const int32_t* post_doc, const uint16_t* post_tf,
                 int64_t n_terms, int64_t nnz, const int32_t* doc_len, int64_t n_docs, double avgdl,
                 const double* idf, int32_t variant, double k1, double b, double delta, int64_t id_base);
int64_t sb_bm25_count(sb_ctx* ctx);
/*
 * GPU index build -- replaces the corpus pass of BM25Retriever.index (reference src/core/retrievers/sparse.py:70-100,
 * where rank_bm25 builds per-doc frequency dicts, df and doc_len in Python).
 *
 * sb_bm25_build_tokens: host token stream flat_tokens[n_tokens] (non-negative raw token ids; doc i is
 * flat_tokens[doc_off[i] : doc_off[i+1]]).  On the device: sort by (token, position), vocabulary = token runs relabelled
 * in FIRST-OCCURRENCE order (rank_bm25's dict insertion order, which its idf sum depends on), term-major CSR postings
 * with docs ascending, tf, doc_len, df.  Returns the number of terms and postings.
 * sb_bm25_build_read: df[n_terms] (term-id order) and the raw token of every term id, for the host-side idf table
 * (math.log bit for bit) and token -> term-id map.  sb_bm25_build_export: the CSR arrays themselves (persistence /
 * sharding); any pointer may be NULL.
 * sb_bm25_build_finish: installs the built CSR as the context's BM25 index with the host-computed idf (same meaning as
 * the arguments of sb_bm25_load); no posting array ever crosses to the host unless exported.
 */
int sb_bm25_build_tokens(sb_ctx* ctx, const int32_t* flat_tokens, int64_t n_tokens, const int64_t* doc_off,
                         int64_t n_docs, int64_t* n_terms_out, int64_t* nnz_out);
int sb_bm25_build_read(sb_ctx* ctx, int64_t* df_out, int32_t* term_token_out);
int sb_bm25_build_export(sb_ctx* ctx, int64_t* indptr_out, int32_t* post_doc_out, uint16_t* post_tf_out,
                         int32_t* doc_len_out);
int sb_bm25_build_finish(sb_ctx* ctx, const double* idf, double avgdl, int32_t variant, double k1, double b,
                         double delta, int64_t id_base);
/*
 * sb_bm25_topk: B queries given as term ids (q_terms, CSR offsets q_off[B+1]; -1 = unknown token; duplicates are
 * scored twice exactly like the reference).  Outputs best-first (score desc, id asc), only score > 0:
 * out_ids[B*k], out_scores[B*k] (bit-identical to the fp64 NumPy arithmetic), out_counts[B] (may be < k).
 */
int sb_bm25_topk(sb_ctx* ctx, const int32_t* q_terms, const int32_t* q_off, int32_t B, int32_t k,
                 int64_t* out_ids, double* out_scores, int32_t* out_counts);
int sb_bm25_topk_dev(sb_ctx* ctx, const int32_t* q_terms_dev, const int32_t* q_off_dev, int32_t B, int32_t n_q_terms,
                     int32_t max_q_len, int32_t k, int64_t* out_ids_dev, double* out_scores_dev,
                     int32_t* out_counts_dev, void* stream);
/* full score vector of ONE query (fp64, n_docs entries) -- bit-exactness checks against get_scores */
int sb_bm25_scores(sb_ctx* ctx, const int32_t* q_terms, int32_t n_q, double* out_scores);

/* ---------------------------------------------------------------- K3: fusion -------------------------------- */
/*
 * Replaces the fusion block of HybridRetriever.retrieve (reference src/core/retrievers/hybrid.py:204-298):
 * rrf / weighted_rrf / comb_sum over a dense list (cache hits already prepended), a sparse list and a
 * retriever-plugin list, optional additive scorer-plugin scores, stable sort, truncate to k.
 *
 * Batched: B queries, each list padded to a fixed stride (d_stride / s_stride / p_stride) with per-query counts.
 * `extra` (may be NULL) holds `n_extra` per-query additive score rows [B][n_extra][e_stride] (one row per scorer
 * plugin, added one after the other like hybrid.py:275-285) indexed by merged-document order
 * (unique dense ids in first-occurrence order, then sparse-only ids; hybrid.py:262-271).
 * rrf_k is a double because Python evaluates `rrf_k + rank` with whatever number type the caller passed.
 * Outputs: out_ids[B*k], out_scores[B*k], out_src[B*k] (bit0: id had a dense doc, bit1: sparse doc; plugin-only ids
 * have out_src == 0 and are dropped by the caller AFTER truncation exactly like hybrid.py:291-298), out_counts[B].
 */
int sb_fuse(sb_ctx* ctx, int32_t method, double rrf_k, double w_dense, double w_sparse, int32_t B,
            const int64_t* d_ids, const double* d_sc, const int32_t* d_n, int32_t d_stride,
            const int64_t* s_ids, const double* s_sc, const int32_t* s_n, int32_t s_stride,
            const int64_t* p_ids, const double* p_sc, const int32_t* p_n, int32_t p_stride,
            const double* extra, int32_t n_extra, int32_t e_stride, int32_t k,
            int64_t* out_ids, double* out_scores, int32_t* out_src, int32_t* out_counts);
int sb_fuse_dev(sb_ctx* ctx, int32_t method, double rrf_k, double w_dense, double w_sparse, int32_t B,
                const int64_t* d_ids, const double* d_sc, const int32_t* d_n, int32_t d_stride,
                const int64_t* s_ids, const double* s_sc, const int32_t* s_n, int32_t s_stride,
                const int64_t* p_ids, const double* p_sc, const int32_t* p_n, int32_t p_stride,
                const double* extra, int32_t n_extra, int32_t e_stride, int32_t k,
                int64_t* out_ids, double* out_scores, int32_t* out_src, int32_t* out_counts, void* stream);

/*
 * sb_hybrid_topk: the whole retrieve -> fuse path of HybridRetriever.retrieve (reference src/core/retrievers/hybrid.py:131-300)
 * for B queries from HOST buffers, single shard: q [B x dim of dense slot 0] fp32, query term ids q_terms / q_off[B+1] as
 * for sb_bm25_topk, fusion parameters as for sb_fuse (no plugin lists).  One H2D of the inputs, K1 + K2 + K3 on the
 * context's stream, one D2H of out_ids / out_scores / out_src [B*k] and out_counts [B].
 */
int sb_hybrid_topk(sb_ctx* ctx, const float* q, const int32_t* q_terms, const int32_t* q_off, int32_t B, int32_t k,
                   int32_t method, double rrf_k, double w_dense, double w_sparse, int64_t* out_ids, double* out_scores,
                   int32_t* out_src, int32_t* out_counts);
/*
 * sb_hybrid_rerank_topk: the same followed by the cross-encoder rerank of rerank_node (reference
 * src/core/graph/nodes.py:138-227 / jina_reranker.py:192-295) on the fused top-k: q_tok [B x lq] word pieces and q_len [B]
 * of the queries (documents come from sb_ce_tokens_load), pairs framed to length S on the device; out_ids / out_scores
 * (sigmoid relevance) [B x k_out], out_counts [B].  One H2D, one D2H.
 */
int sb_hybrid_rerank_topk(sb_ctx* ctx, const float* q, const int32_t* q_terms, const int32_t* q_off, const int32_t* q_tok,
                          const int32_t* q_len, int32_t lq, int32_t B, int32_t k, int32_t k_out, int32_t S, int32_t method,
                          double rrf_k, double w_dense, double w_sparse, int64_t* out_ids, float* out_scores,
                          int32_t* out_counts);

/* ---------------------------------------------------------------- K4: semantic similarity + MMR ------------- */
/*
 * Replaces SemanticSimilarityScorer.score and MMRScorer.score (reference src/core/retrievers/scorers.py:152-191,
 * 222-273).  q[d] and cand[n*d] are fp32 host embeddings (what embed_sync / embed_many_sync returned); if `cand`
 * is NULL the candidates are taken from dense slot `slot` by id (cand_ids[n]) -- the stored corpus vectors.
 * out_sem[n] = w_sem * cos(q, d_i) (0 if either norm is 0); out_mmr[n] = greedy-MMR scores with the reference's
 * quirks (strict '>' argmax from -1.0, first index wins ties, never-selected-or-zero -> rel*w*lambda, clip at 0).
 * Either output pointer may be NULL.
 */
int sb_semantic_mmr(sb_ctx* ctx, int slot, const float* q, int32_t d, const float* cand, const int64_t* cand_ids,
                    int32_t n, double w_sem, double lambda, double w_mmr, double* out_sem, double* out_mmr);

/* ---------------------------------------------------------------- K5: cross-encoder rerank ------------------ */
/*
 * Replaces the remote Jina rerank call behind JinaReranker.rerank (reference
 * src/core/rerankers/jina_reranker.py:139-144,255-276) with a local BERT-style sequence classifier
 * (MiniLM-L6 shape by default: 6 layers, hidden 384, 12 heads, FFN 1536, vocab 30522, max_pos 512, 1 label).
 */
typedef struct sb_ce_config {
  int32_t vocab_size;
  int32_t hidden;
  int32_t layers;
  int32_t heads;
  int32_t intermediate;
  int32_t max_pos;
  int32_t type_vocab;
  float ln_eps;
} sb_ce_config;
/*
 * weights: one contiguous fp32 host blob in the order documented in sentio_b200/cross_encoder.py
 * (word/pos/type embeddings, emb LN, per layer {Wq,bq,Wk,bk,Wv,bv,Wo,bo,LN1,W1,b1,W2,b2,LN2}, pooler W,b,
 * classifier w,b); n_floats is checked against the config.
 */
int sb_ce_load(sb_ctx* ctx, const float* weights, int64_t n_floats, const sb_ce_config* cfg);
/*
 * input_ids / token_type: P x S int32 (host), lengths[P] = number of real tokens per pair (attention mask); positions
 * >= lengths[p] are padding and are skipped entirely (tokens are packed on the device; same [CLS] logit as masking).
 * out_logits[P], out_sigmoid[P] (relevance in [0,1], reference test_jina_reranker.py:283-300).
 */
int sb_ce_score(sb_ctx* ctx, const int32_t* input_ids, const int32_t* token_type, const int32_t* lengths,
                int32_t P, int32_t S, float* out_logits, float* out_sigmoid);
int sb_ce_score_dev(sb_ctx* ctx, const int32_t* input_ids_dev, const int32_t* token_type_dev,
                    const int32_t* lengths_dev, int32_t P, int32_t S, float* out_logits_dev,
                    float* out_sigmoid_dev, void* stream);

/*
 * Query / document embedder on the device (SURVEY 8f row 1) -- replaces the remote `embedder.embed_sync(query)` that
 * precedes the dense search in DenseRetriever.retrieve (reference src/core/retrievers/dense.py:43; the provider is the
 * hosted Jina embeddings API, src/core/embeddings/providers/jina.py).  A second BERT-style encoder (same blob layout and
 * kernels as the cross-encoder; its pooler / classifier tensors are ignored) whose final [CLS] state is optionally
 * projected (proj_w [out_dim, hidden], proj_b [out_dim], fp32; NULL = identity) and L2-normalised.
 * sb_enc_embed: input_ids / token_type P x S int32 (host), lengths[P]; out[P * sb_enc_dim()] fp32 (host).
 * sb_enc_embed_dev: the same on device buffers (chains straight into sb_dense_topk_dev without a host round trip).
 */
int sb_enc_load(sb_ctx* ctx, const float* weights, int64_t n_floats, const sb_ce_config* cfg, const float* proj_w,
                const float* proj_b, int32_t out_dim);
int32_t sb_enc_dim(sb_ctx* ctx);
int sb_enc_embed(sb_ctx* ctx, const int32_t* input_ids, const int32_t* token_type, const int32_t* lengths, int32_t P,
                 int32_t S, int32_t normalize, float* out);
int sb_enc_embed_dev(sb_ctx* ctx, const int32_t* input_ids_dev, const int32_t* token_type_dev,
                     const int32_t* lengths_dev, int32_t P, int32_t S, int32_t normalize, float* out_dev, void* stream);

/*
 * Work counters of the packed-token forward since the last reset: out3 = {pairs scored, sum of pair lengths (token rows
 * actually computed), sum of squared pair lengths}.  flops = layers * (24 * H^2 * out3[1] + 4 * H * out3[2]) -- used by
 * bench.py so the tensor-pipe roofline counts the work done, not the padding skipped.  Synchronises the device.
 */
int sb_ce_stats(sb_ctx* ctx, int64_t* out3, int32_t reset);

/*
 * Batched rerank (retrieve -> rerank without leaving the device): sb_ce_tokens_load stores the shard's pre-tokenised
 * documents (doc i = doc_tok[i][0..doc_len[i]), word-piece ids < 65536, id = id_base + i).  sb_rerank_dev frames
 * `[CLS] query [SEP] doc [SEP]` for every (query b, candidate j < cand_cnt[b]) pair on the device, runs the cross-encoder
 * and emits, per query, the k_out candidates with the highest relevance (stable on the incoming order, like the
 * reference's sorted(..., reverse=True) at jina_reranker.py:279-283): out_ids[B*k_out], out_scores[B*k_out] (sigmoid),
 * out_counts[B].
 */
int sb_ce_tokens_load(sb_ctx* ctx, const uint16_t* doc_tok, const int32_t* doc_len, int64_t n_docs, int32_t ld,
                      int64_t id_base);
int sb_rerank_dev(sb_ctx* ctx, const int32_t* q_tok_dev, const int32_t* q_len_dev, int32_t lq,
                  const int64_t* cand_ids_dev, const int32_t* cand_cnt_dev, int32_t B, int32_t k, int32_t S,
                  int32_t k_out, int64_t* out_ids_dev, float* out_scores_dev, int32_t* out_counts_dev, void* stream);

/*
 * Test hook for the tcgen05 GEMM inside K5: out[M,N] = epilogue(A[M,K] * W[N,K]^T + bias (+ residual)), operands given as
 * host fp32 and rounded to fp16 on the device; epi 0 = bias (fp16 result), 1 = bias + erf-GELU (fp16 result),
 * 2 = bias + residual (fp32 result).  N % 128 == 0, K % 64 == 0.
 */
int sb_ce_gemm_test(sb_ctx* ctx, const float* a, const float* w, const float* bias, const float* residual, int32_t M,
                    int32_t N, int32_t K, int32_t epi, float* out);

/* ---------------------------------------------------------------- K6: shard merge ---------------------------- */
/*
 * Multi-GPU: after ONE all-gather of per-shard top-k records, every rank merges G shard lists per query into the
 * global top-k (score desc, id asc).  The pointers address shard 0's ids [B][k] / scores [B][k] / counts [B]; shard g's
 * copies start `shard_stride_bytes * g` bytes later (= the per-rank record size of the gathered buffer).
 */
int sb_merge_shards_dev(sb_ctx* ctx, const int64_t* in_ids, const double* in_scores, const int32_t* in_counts,
                        int64_t shard_stride_bytes, int32_t G, int32_t B, int32_t k, int64_t* out_ids,
                        double* out_scores, int32_t* out_counts, void* stream);

/* ---------------------------------------------------------------- K7: document selector ------------------------ */
/*
 * Batched form of select_documents_node (reference src/core/graph/nodes.py:272-337), the node that follows the reranker:
 * per query, stable sort of the candidates by score (descending), repeated ids dropped, the first top_k unique documents
 * walked, blank documents skipped, documents kept while the running `len(text) // 4` token estimate stays <= max_tokens
 * (the first document that does not fit ends the walk).
 * sb_doc_chars_load: n_chars[i] = characters of document (id_base + i)'s usable text -- `doc.text`, else
 * `metadata["content"]` (nodes.py:296-299) -- and 0 for a blank one.
 * sb_select_dev: cand_ids [B,k] / cand_scores [B,k] (score_dtype 0 = float32, e.g. sb_rerank_dev's output, 1 = float64,
 * e.g. sb_fuse_dev's) / cand_cnt [B] -> out_ids [B,top_k] (-1 padded), out_scores [B,top_k] (same dtype),
 * out_counts [B] (= metadata.selected_count), out_tokens [B] (= metadata.selected_tokens).
 */
int sb_doc_chars_load(sb_ctx* ctx, const int32_t* n_chars, int64_t n_docs, int64_t id_base);
int sb_select_dev(sb_ctx* ctx, const int64_t* cand_ids_dev, const void* cand_scores_dev, int32_t score_dtype,
                  const int32_t* cand_cnt_dev, int32_t B, int32_t k, int32_t top_k, int32_t max_tokens,
                  int64_t* out_ids_dev, void* out_scores_dev, int32_t* out_counts_dev, int32_t* out_tokens_dev,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SENTIO_B200_H */
