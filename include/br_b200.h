/* br_b200.h - C ABI of the B200-native BM25 / cosine retrieval hot path.
 *
 * The reference (Harkeerat2002/document-retrieval) has no FFI layer: its boundary for this path is
 * a set of Python callables (SURVEY 8b).  This header is the boundary a binding for those
 * callables sits on; document_retrieval_b200/_lib.py is that binding (ctypes) and INTEGRATION.md
 * shows the stub a reference maintainer would add.  Each entry point names the reference code it
 * replaces (file:line in the reference checkout; .ipynb lines are raw JSON lines).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; every function returns 0 on success and a negative
 *     br_status on failure; br_last_error() gives the message (thread-local).
 *   - "dev" pointers are CUDA device pointers on the handle's device, caller-owned unless stated;
 *     "host" pointers are ordinary host memory.  Work is enqueued on the cudaStream_t passed as
 *     `stream` (an opaque void* here so that C callers need no CUDA headers); calls that must
 *     return host-visible values synchronise that stream before returning.
 *   - One handle = one device.  A handle is not thread-safe; distinct handles are independent.
 *   - Doc ids are 32-bit and local to the handle's shard: global id = doc_base + local id.
 *   - There is no CPU fallback anywhere behind this interface.
 */
#ifndef BR_B200_H
#define BR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct br_index br_index;

typedef enum br_status {
    BR_OK = 0,
    BR_ERR_INVALID = -1,   /* bad argument (null pointer, token id outside [0,vocab), k out of range ...) */
    BR_ERR_CUDA = -2,      /* a CUDA runtime call or kernel failed */
    BR_ERR_STATE = -3,     /* call order violated (e.g. query before br_index_finalize) */
    BR_ERR_UNSUPPORTED = -4
} br_status;

/* BM25 formula variants (SURVEY appendix A):
 *   NOTEBOOK        idf = ln(1+(N-df+.5)/(df+.5)), norm = 1-b+dl/avgdl      bm25_ranking.ipynb:189,202
 *   OKAPI           same idf,                       norm = 1-b+b*dl/avgdl   team_run1.py:187,193
 *   OKAPI_NO_PLUS1  idf = ln((N-df+.5)/(df+.5)),    norm = 1-b+b*dl/avgdl   cosine_similarity_bm25_reranking.py:179 */
typedef enum br_variant { BR_NOTEBOOK = 0, BR_OKAPI = 1, BR_OKAPI_NO_PLUS1 = 2 } br_variant;

const char* br_last_error(void);
/* "br_b200 <version> sm_100a" */
const char* br_version(void);

/* ---------------------------------------------------------------------------------------------
 * Index build.  Replaces BM25.__init__/build (bm25_ranking.ipynb:167-189,
 * final_implementation.py:92-118), compute_tf_df_and_avgdl
 * (cosine_similarity_bm25_reranking.py:129-172) and build_inverted_index (team_run1.py:80-99).
 *
 * Phase 1 (br_index_build): tokenised docs -> CSR posting lists sorted by (term, doc) with raw tf,
 * per-doc length dl and the shard-local df histogram.  token_ids_dev is int32[doc_offsets[n_docs]],
 * doc_offsets_dev is int64[n_docs+1]; both are only read and may be freed after the call.
 * Phase 2 (br_index_finalize): fixes the corpus statistics the weights depend on - N, sum of
 * doc lengths and the df histogram.  A single-GPU caller passes n_stat = 0, sum_dl_stat = 0,
 * df_stat_host = NULL (the shard's own statistics are used).  A doc-sharded caller all-reduces
 * (sum) br_index_df_dev()/n_docs/sum_dl across ranks between the two phases and passes the
 * global values, so every shard computes bit-identical idf / avgdl.  idf is evaluated on the host
 * in float64 with libm log() - the same routine CPython's math.log uses
 * (bm25_ranking.ipynb:189) - and each posting gets w = fp32(idf*((tf*(k1+1))/(tf+k1*norm))).
 * ------------------------------------------------------------------------------------------- */
int br_index_build(const int32_t* token_ids_dev, const int64_t* doc_offsets_dev, int64_t n_docs,
                   int32_t vocab, int64_t doc_base, void* stream, br_index** out);
int br_index_finalize(br_index* ix, double k1, double b, int variant, double n_stat,
                      double sum_dl_stat, const int64_t* df_stat_host, void* stream);
void br_index_destroy(br_index* ix);

/* Append n_docs documents to a built index.  token_ids_dev / doc_offsets_dev: the same layout as br_index_build.
 * vocab is the new vocabulary size, >= the handle's; token ids must be in [0, vocab).  The appended docs get local ids
 * n_docs_old .. n_docs_old + n_docs - 1.  On success the handle is NOT finalised: every query entry point returns
 * BR_ERR_STATE until br_index_finalize is called again (N, avgdl and df changed, so every weight changes).
 * On any error the handle is left exactly as it was, including its finalised state, and still answers queries with the
 * same results.
 * Appending B to the index of A and finalising gives the same bits as building A followed by B from scratch and
 * finalising: the same CSR, df, idf, weights, skip tables and dense rows, hence the same results from every query.
 * Works on any handle (built, imported, loaded from an index file); doc_base is kept.  n_docs < 1, vocab below the
 * handle's, a token id outside [0, vocab) or decreasing offsets: BR_ERR_INVALID.  A term occurring more than 65535
 * times in one doc, or a grown index of 2^31 docs, 2^32 tokens or 2^32 postings or more: BR_ERR_UNSUPPORTED.  A
 * doc-sharded caller re-finalises every shard with the all-reduced statistics afterwards. */
int br_index_append(br_index* ix, const int32_t* token_ids_dev, const int64_t* doc_offsets_dev, int64_t n_docs,
                    int32_t vocab, void* stream);

/* Remove documents from a built index.  remove_dev is uint8[n_docs] on the device; a nonzero byte removes that local doc.
 * The kept docs keep their order: a kept doc's new local id is its rank among the kept docs (old id kept[i] becomes i,
 * kept = the ids with a zero byte, ascending).  doc_base, term ids and vocab do not change; a term that loses every
 * posting keeps its id with df 0, like an id no doc uses in br_index_build.  On success the handle is NOT finalised:
 * every query entry point returns BR_ERR_STATE until br_index_finalize is called again (N, avgdl and df changed).
 * Removing R from the index of C and finalising gives the same bits as building the docs of C not in R, in order, over
 * the same vocab and finalising: the same CSR, df, idf, weights, skip tables and dense rows, hence the same results from
 * every query.
 * No nonzero byte: BR_OK, and the handle is left as it was, still finalised.  Null pointers or a mask that removes every
 * doc: BR_ERR_INVALID.  On any error the handle is left exactly as it was, including its finalised state, and still
 * answers queries with the same results.  Works on any handle (built, imported, appended to).  A doc-sharded caller
 * re-finalises every shard with the all-reduced statistics afterwards. */
int br_index_remove(br_index* ix, const uint8_t* remove_dev, void* stream);

/* corpus_size / nnz / avgdl / sum(dl) attributes (bm25_ranking.ipynb:170-171). Any out may be NULL. */
int br_index_stats(const br_index* ix, int64_t* n_docs, int32_t* vocab, int64_t* nnz,
                   double* avgdl, int64_t* sum_dl, int64_t* doc_base);
/* The corpus statistics the weights were computed with (br_index_finalize's n_stat / sum_dl_stat after defaulting):
 * differ from br_index_stats for a doc shard.  Stored in the flat index file so that a shard can be re-finalised. */
int br_index_stats_in_force(const br_index* ix, double* n_stat, double* sum_dl_stat);
/* Device pointer to the shard-local df histogram, uint32[vocab] (for the cross-shard all-reduce). */
const uint32_t* br_index_df_dev(const br_index* ix);
/* `df` / `idf` attributes (bm25_ranking.ipynb:173-174,188-189; compute_idf
 * cosine_similarity_bm25_reranking.py:176-182): df_host int64[vocab] (statistics in force),
 * idf_host double[vocab] (NaN where df == 0).  Either may be NULL. */
int br_index_export_df_idf(const br_index* ix, int64_t* df_host, double* idf_host);
/* CSR export for `inverted_index` / `term_freqs` / `doc_lengths` attributes and for pickling
 * (joblib.dump(bm25_model, ...), bm25_ranking.ipynb:312).  row_ptr_host int64[vocab+1],
 * doc_host int32[nnz], tf_host int32[nnz], dl_host int32[n_docs]; any may be NULL. */
int br_index_export_csr(const br_index* ix, int64_t* row_ptr_host, int32_t* doc_host,
                        int32_t* tf_host, int32_t* dl_host);
/* Rebuild a handle from an exported CSR (unpickling). Call br_index_finalize afterwards. */
int br_index_import_csr(const int64_t* row_ptr_host, const int32_t* doc_host, const int32_t* tf_host,
                        const int32_t* dl_host, int64_t n_docs, int32_t vocab, int64_t doc_base,
                        void* stream, br_index** out);

/* The same two with DEVICE arrays and 16-bit tf - the path of the flat index file (BM25.save / BM25.load): the file's
 * arrays are staged through pinned host memory straight into device buffers, no host-side copy or conversion.  This
 * is what replaces the joblib model files whose loading dominated the reference's run time (bm25_ranking.ipynb:222-251,
 * final_implementation.py:187-287).  Import validates the CSR on the device (row_ptr a monotone [0 .. nnz] offset array,
 * doc ids in range and strictly ascending inside a posting list, 1 <= tf <= 65535, doc lengths >= 0) and fails with
 * BR_ERR_INVALID otherwise; br_index_import_csr goes through the same checks.  Call br_index_finalize afterwards. */
int br_index_export_csr_dev(const br_index* ix, int64_t* row_ptr_dev, int32_t* doc_dev, uint16_t* tf_dev,
                            int32_t* dl_dev, void* stream);
int br_index_import_csr_dev(const int64_t* row_ptr_dev, const int32_t* doc_dev, const uint16_t* tf_dev,
                            const int32_t* dl_dev, int64_t n_docs, int32_t vocab, int64_t nnz, int64_t doc_base,
                            void* stream, br_index** out);

/* ---------------------------------------------------------------------------------------------
 * Queries.  A batch is CSR-packed term ids: q_terms_dev int32[q_offsets[nq]], q_offsets_dev
 * int32[nq+1], device memory.  Term ids outside [0,vocab) or with no postings are skipped, like
 * `if word not in self.idf: continue` (bm25_ranking.ipynb:195-196).
 * dedup != 0: set(query) semantics (bm25_ranking.ipynb:193); dedup == 0: every occurrence counts,
 * in query order (team_run1.py:183).
 * ------------------------------------------------------------------------------------------- */

/* Replaces BM25.get_scores (bm25_ranking.ipynb:191-204) / calculate_scores
 * (final_implementation.py:127-145) for a batch: out_scores_dev float32[nq, n_docs] (fp32
 * accumulation of the precomputed posting weights: per doc, |fp32 - float64 reference| <=
 * (n + 2) * 2^-24 * sum_t mult_t * |w_t,d| over the query's n distinct terms with multiplicity mult_t
 * and float64 weights w_t,d; for weights of one sign that is within 1e-5 relative, while under
 * okapi_no_plus1 a query with a term of negative idf can cancel to an fp32 0 of a non-zero score). */
int br_score_batch(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev,
                   int32_t nq, int dedup, float* out_scores_dev, void* stream);

/* Replaces BM25.retrieve_top_n (bm25_ranking.ipynb:206-213), retrieve_top_n_batch
 * (final_implementation.py:179-181) and score_documents_for_query's nlargest
 * (team_run1.py:196) for a batch.  Outputs are [nq, k], best first, ordered by (float64 score
 * descending, doc id ascending): out_ids_dev int32 (local ids; -1 pads a short result),
 * out_scores_dev double (exact float64 re-evaluation of the reference formula, terms summed in
 * ascending term id for dedup != 0 and in query order otherwise), out_counts_dev int32[nq]
 * (number of valid entries; may be NULL).  positive_only != 0 keeps only docs whose float64 score
 * is not 0 (team_run1.py:196 ranks the docs with a hit; a doc whose only hits are terms of idf 0 -
 * df = N/2 under okapi_no_plus1 - scores exactly 0 and is dropped too); otherwise zero-score docs
 * fill the tail in doc-id order like the dense argpartition (bm25_ranking.ipynb:211).
 * 1 <= k <= BR_MAX_K.
 * The call synchronises `stream` before returning. */
/* n_terms = q_offsets[nq], the number of term slots of the batch, which the caller knows from packing it (an upper
 * bound works too); pass -1 when it is unknown - the library then reads it back from the device, which costs a
 * stream synchronisation before any kernel of the batch is launched.  q_offsets running past n_terms is
 * BR_ERR_INVALID. */
#define BR_MAX_K 1024
int br_topk_batch(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev,
                  int32_t nq, int32_t n_terms, int32_t k, int dedup, int positive_only, int32_t* out_ids_dev,
                  double* out_scores_dev, int32_t* out_counts_dev, void* stream);
/* The same with the result as packed records {global doc id = doc_base + local id (-1 pads), float64 score}
 * [nq, k]: the unit a doc-sharded caller all-gathers (one collective instead of two, SURVEY 8e). */
typedef struct br_record {
    int64_t id;
    double score;
} br_record;
int br_topk_batch_records(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                          int32_t n_terms, int32_t k, int dedup, int positive_only, br_record* out_records_dev,
                          int32_t* out_counts_dev, void* stream);

/* Filtered top-k: restrict what a query may return to an allow-list of docs (one language, one tenant, a date range,
 * "not deleted").  A filter is a set of bitmap rows over the handle's LOCAL doc ids; every query selects one row or none.
 *   bits_dev       uint32[n_rows, words], device: bit (d & 31) of word (d >> 5) of row f set = local doc d may be
 *                  returned by a query that uses row f; bits at d >= n_docs are ignored
 *   words          row stride in words, >= ceil(n_docs / 32)
 *   query_row_dev  int32[nq], device: the row query q uses, -1 = unfiltered; NULL = row 0 for every query
 * The result of a filtered query is the unfiltered call's result on the corpus restricted to its allowed docs: doc ids,
 * N, avgdl, df and idf are unchanged (scores are bit-identical to the unfiltered scores of the same docs), the order is
 * (float64 score desc, doc id asc), positive_only == 0 fills a short tail with allowed zero-score docs in doc-id order,
 * and a query with fewer than k allowed docs gets -1 padding (out_counts = number of valid entries).  An all-ones row
 * gives exactly the unfiltered result.  A null bits pointer, words < ceil(n_docs / 32) or n_rows < 1 is BR_ERR_INVALID;
 * a query_row value outside [-1, n_rows) is detected on the device, never used to address the bitmap, and reported as
 * BR_ERR_INVALID when the call returns.  filter == NULL: the unfiltered call.  The filter's arrays are only read. */
typedef struct br_doc_filter {
    const uint32_t* bits_dev;
    int64_t words;
    int32_t n_rows;
    const int32_t* query_row_dev;
} br_doc_filter;
int br_topk_batch_filtered(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                           int32_t n_terms, int32_t k, int dedup, int positive_only, int32_t* out_ids_dev,
                           double* out_scores_dev, int32_t* out_counts_dev, const br_doc_filter* filter, void* stream);
int br_topk_batch_records_filtered(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                                   int32_t n_terms, int32_t k, int dedup, int positive_only, br_record* out_records_dev,
                                   int32_t* out_counts_dev, const br_doc_filter* filter, void* stream);

/* Exact float64 BM25 of explicit (query, doc) pairs - the arithmetic of the loop body at
 * bm25_ranking.ipynb:199-203 / team_run1.py:188-194 evaluated doc-at-a-time: query q owns the
 * candidate docs cand_ids_dev[cand_off_dev[q] .. cand_off_dev[q+1]) (local ids, int32; cand_off
 * int64[nq+1]); out_scores_dev double[cand_off[nq]].  Used for full rankings (n >= N,
 * bm25_ranking.ipynb:208-209) and for re-scoring externally chosen candidates. */
int br_rescore_docs(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                    int dedup, const int32_t* cand_ids_dev, const int64_t* cand_off_dev,
                    double* out_scores_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Sparse TF-IDF cosine -> BM25 re-rank (implementation 2 of the reference,
 * cosine_similarity_bm25_reranking.py:198-238).  Needs an index finalised with BR_OKAPI_NO_PLUS1
 * (compute_idf has no +1, :179).
 * ------------------------------------------------------------------------------------------- */
/* Build the second weight table w' = tf*idf^2/||d||, ||d|| = L2 norm of the doc's tf*idf vector
 * (create_tfidf_embedding :72-110, doc_norms :210-211).  Idempotent. */
int br_index_enable_tfidf(br_index* ix, void* stream);
/* First stage: top-k docs by TF-IDF cosine against the query vector "idf per distinct in-corpus term"
 * (generate_query_embedding :121-126).  The fp32 accumulation of w' only selects a candidate band; every band
 * member is re-scored in float64 with the reference's mixed precision (float32 tf*idf entries, float64 doc norms,
 * float32 normalised query, float64 products, :88,210-226), so the top-k SET is the reference's wherever its own
 * order is defined.  out_scores_dev double[nq,k] = that cosine; order (cosine desc, doc id asc); zero-cosine docs
 * fill a short tail in doc order like the full argsort (:229).  Synchronises `stream`. */
int br_tfidf_cosine_topk(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                         int32_t k, int32_t* out_ids_dev, double* out_scores_dev, int32_t* out_counts_dev,
                         void* stream);
/* bm25_score (cosine_similarity_bm25_reranking.py:185-195) for explicit (query, doc) pairs, float64:
 * doc_length = sum of the query terms' tf in the doc (:187), duplicates counted, idf from the index.
 * Same candidate layout as br_rescore_docs. */
int br_rerank_v3_scores(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                        const int32_t* cand_ids_dev, const int64_t* cand_off_dev, double* out_scores_dev,
                        void* stream);

/* Threshold sharing between the shards of a doc-sharded index.  The tiled scorer prunes with a running lower bound
 * thr[q] of each query's k-th best score.  A shard alone learns it from its own docs only - from 1/N of the corpus, so its
 * launches run with the loose thresholds the single index only has in its first tiles.  With this callback set (k <= 32),
 * the library calls fn(local_dev, gathered_dev, n_floats, stream, user) once after its threshold seeding (local = thr[nq])
 * and once after each of the first `rounds` tile launches of a batch (local = the shard's current k best fp32 scores of
 * every query, float[nq, k], zero-padded); fn must ALL-GATHER the n_floats floats of every shard into
 * gathered_dev float[world, n_floats] (an NCCL all-gather enqueued on `stream`; return 0).  The library then raises
 * thr[q] to the maximum of the shards' seeds / to the k-th largest of the world x k gathered scores: k distinct docs of the
 * WHOLE corpus score at least that much, which is all the merge needs; a shard may then return fewer than k docs for a
 * query.  Every shard must use the same `rounds` (at most br_tile_launch_count - 1 of the smallest shard) and `world`, so
 * that all of them make the same calls per batch; fn == NULL or rounds < 0 switches the exchange off.  sharded.py's
 * ShardedBM25 sets this up. */
typedef int (*br_thr_exchange_fn)(const float* local_dev, float* gathered_dev, int64_t n_floats, void* stream, void* user);
int br_set_thr_exchange(br_index* ix, br_thr_exchange_fn fn, void* user, int rounds, int world);
/* Tile-kernel launches a batch with this k makes on this index (0: the tiled path does not apply). */
int br_tile_launch_count(const br_index* ix, int32_t k);

/* Merge of per-shard top-k lists after the all-gather (no reference analogue: the reference is
 * single-process).  ids_dev int64[n_parts, nq, k] (global ids, -1 = padding), scores_dev
 * double[n_parts, nq, k]; outputs [nq, k] ordered by (score desc, id asc). */
int br_topk_merge(const int64_t* ids_dev, const double* scores_dev, int32_t n_parts, int32_t nq,
                  int32_t k, int64_t* out_ids_dev, double* out_scores_dev, void* stream);
/* The same over the all-gathered records of br_topk_batch_records: records_dev br_record[n_parts, nq, k]. */
int br_topk_merge_records(const br_record* records_dev, int32_t n_parts, int32_t nq, int32_t k,
                          int64_t* out_ids_dev, double* out_scores_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dense cosine similarity on bf16 embeddings.  Replaces the re-rank block of team_run1.py:269-295
 * (e/(||e||+1e-10) on both sides, torch.matmul, torch.topk) and faiss.IndexFlatIP on normalised
 * vectors (faiss_based_ANN_Implementation.py:279-283).  Embeddings are row-major bf16 [n, d], d a
 * multiple of 8, 16-byte aligned, NOT pre-normalised; scores are fp32.
 * ------------------------------------------------------------------------------------------- */
/* out_inv_norm_dev[i] = 1 / (||emb[i]||_2 + 1e-10)  (.norm() + 1e-10, team_run1.py:271,276). */
int br_row_inv_norms(const void* emb_bf16_dev, int64_t n, int32_t d, float* out_inv_norm_dev, void* stream);
/* Exact brute-force top-k (1 <= k <= 256) of every query over all docs: bf16 tcgen05 GEMM with the
 * normalisation and the top-k filter fused into the epilogue.  doc_inv_norm_dev from
 * br_row_inv_norms (computed once per corpus).  Outputs [nq, k], best first, ties by doc id:
 * out_ids_dev int64 (doc_base + local row, -1 pads), out_sims_dev float.  A query for which one launch finds more
 * than 1024 rows at or above its running threshold (masses of duplicate embeddings, or rows ordered by similarity to
 * the queries) is answered exactly by a full gather pass instead of the filter - any number of such queries, 64 per
 * pass; slower, never wrong.  nq = 0 returns at once (queries and outputs may then be NULL).  Synchronises `stream`. */
int br_cosine_topk(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_docs, int32_t d,
                   const void* queries_bf16_dev, int32_t nq, int32_t k, int64_t doc_base,
                   int64_t* out_ids_dev, float* out_sims_dev, void* stream);
/* The same restricted to per-query allow-lists of rows (br_doc_filter over the local rows 0..n_docs-1, same rules as
 * br_topk_batch_filtered): a filtered query's result is br_cosine_topk over its allowed rows only - exact, no
 * over-fetch; fewer than k allowed rows pad with -1.  filter == NULL: br_cosine_topk. */
int br_cosine_topk_filtered(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_docs, int32_t d,
                            const void* queries_bf16_dev, int32_t nq, int32_t k, int64_t doc_base,
                            int64_t* out_ids_dev, float* out_sims_dev, const br_doc_filter* filter, void* stream);
/* Grouped (document-level) cosine top-k, e.g. documents ranked by the best of their sentence embeddings ("max-sim").
 * Embedding row r belongs to group row_group_dev[r] (int32[n_rows], device, non-decreasing, values in [0, n_groups): a
 * group's rows are one contiguous run, e.g. a document's sentences in order).  A group's score is the largest cosine of
 * its rows, computed exactly as br_cosine_topk computes a row's cosine.  Outputs [nq, k], best first, ordered by
 * (score desc, group id asc): out_ids_dev int64 = doc_base + group id, -1 pads when fewer than k non-empty groups
 * (allowed groups, with a filter) exist; out_sims_dev float.  Groups without rows are never returned.  1 <= k <= 256.
 * filter (may be NULL): a br_doc_filter over GROUP ids (words >= ceil(n_groups / 32)), same rules as
 * br_cosine_topk_filtered.  A decreasing or out-of-range row_group is BR_ERR_INVALID (checked on the device before any
 * scoring).  A query whose candidate lists overflow takes the exact gather pass as in br_cosine_topk (d <= 1024).
 * Synchronises `stream`. */
int br_cosine_topk_grouped(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_rows, int32_t d,
                           const int32_t* row_group_dev, int32_t n_groups, const void* queries_bf16_dev, int32_t nq,
                           int32_t k, int64_t doc_base, int64_t* out_ids_dev, float* out_sims_dev,
                           const br_doc_filter* filter, void* stream);
/* Process-wide test switch of br_cosine_topk: name = "kernel" (0 auto: query-stationary CTA pairs for d <= 768, else
 * 2-CTA multicast; 1 always multicast).  Both kernels return bit-identical results.  Any other name: BR_ERR_INVALID. */
int br_set_cosine_option(const char* name, int value);
/* Re-rank: query q against its own candidates cand_ids_dev[q, 0..c) (local rows, -1 = empty slot),
 * e.g. the BM25 top-1000 (text_preprocessing_and_embedding_setup.py:342).  doc_inv_norm_dev may be
 * NULL (norms are then computed on the fly, bit-identical to br_row_inv_norms).  Outputs [nq, k] (k <= BR_MAX_K):
 * out_ids_dev int32, out_sims_dev float, ordered by (cosine desc, doc id asc); a candidate repeated in a row is returned
 * once; fewer than k distinct candidates pad with -1 / 0.0.  A candidate id outside [-1, n_docs) is BR_ERR_INVALID (its
 * row is never read).  nq = 0 returns at once (queries, candidates and outputs may then be NULL).  Synchronises
 * `stream`. */
int br_cosine_rerank(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_docs, int32_t d,
                     const void* queries_bf16_dev, int32_t nq, const int32_t* cand_ids_dev, int32_t c,
                     int32_t k, int32_t* out_ids_dev, float* out_sims_dev, void* stream);
/* Grouped re-rank, e.g. BM25's candidate documents re-ranked by the best of their sentence embeddings.  row_group_dev and
 * n_groups as in br_cosine_topk_grouped (non-decreasing, values in [0, n_groups)); doc_inv_norm_dev (br_row_inv_norms) is
 * required.  cand_groups_dev int32[nq, c] holds each query's candidate GROUPS (local group ids, -1 = empty slot); c >= 1,
 * any size.  A group scores the largest cosine of its rows, each computed bit for bit as br_cosine_rerank computes it.
 * Outputs [nq, k] (1 <= k <= BR_MAX_K): out_ids_dev int32 local group ids, out_sims_dev float, ordered by (score desc,
 * group id asc); a group repeated in a row is returned once, groups without rows are never returned, and fewer than k
 * distinct non-empty candidates pad with -1 / 0.0.  A decreasing or out-of-range row_group is BR_ERR_INVALID (checked on
 * the device before any row is read); so is a candidate id outside [-1, n_groups) (never used to find rows, reported at
 * the synchronisation).  d not a multiple of 8 or d > 1024: BR_ERR_UNSUPPORTED.  nq = 0 returns at once (queries,
 * candidates and outputs may then be NULL).  Synchronises `stream`. */
int br_cosine_rerank_grouped(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_rows, int32_t d,
                             const int32_t* row_group_dev, int32_t n_groups, const void* queries_bf16_dev, int32_t nq,
                             const int32_t* cand_groups_dev, int32_t c, int32_t k, int32_t* out_ids_dev,
                             float* out_sims_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Hybrid retrieval: one ranking from a BM25 candidate list and a dense cosine candidate list per query.
 * bm25_ids_dev int32[nq, nb] and dense_ids_dev int32[nq, nd] hold LOCAL doc ids of the BM25 index, -1 = an empty slot
 * (anywhere in a list).  A doc's rank in a list is 1 + the slot of its first occurrence; later repeats are ignored and
 * empty slots do not renumber the slots after them.  The union is the set of distinct valid ids of both lists.
 * 0 <= nb, nd <= BR_MAX_K, nb + nd >= 1, 1 <= k <= BR_MAX_K.  Outputs [nq, k]: the top k union members by (fused score
 * desc, doc id asc), out_ids_dev int32 (-1 pads when the union has fewer than k members), out_scores_dev double (0.0
 * pads), out_counts_dev int32[nq] = valid entries (may be NULL).  An id outside [-1, n_docs) is BR_ERR_INVALID: it is
 * detected on the device and never used to address anything.  nq = 0 returns at once (lists and outputs may then be
 * NULL).  Both calls synchronise `stream`.
 * ------------------------------------------------------------------------------------------- */
/* Reciprocal rank fusion: f(d) = w_bm25 / (rrf_c + r_b(d)) + w_dense / (rrf_c + r_d(d)), a term omitted when d is not in
 * that list; float64, one correctly rounded division per term and one addition (a numpy restatement gives the same
 * bits).  rrf_c >= 0 (60 is usual), w_bm25, w_dense >= 0 and not both 0, all finite; BR_ERR_INVALID otherwise. */
int br_fuse_rrf(const int32_t* bm25_ids_dev, int32_t nb, const int32_t* dense_ids_dev, int32_t nd, int64_t n_docs,
                int32_t nq, double rrf_c, double w_bm25, double w_dense, int32_t k, int32_t* out_ids_dev,
                double* out_scores_dev, int32_t* out_counts_dev, void* stream);
/* Linear fusion of min-max-normalised exact scores: f = alpha * n_b + (1 - alpha) * n_c, alpha in [0, 1].
 *   s_b(d): float64 BM25 of d for the query (q_terms_dev / q_offsets_dev / n_terms / dedup as in br_topk_batch),
 *           bit-identical to br_rescore_docs and to the scores br_topk_batch returns; 0.0 when no query term matches.
 *   s_c(d): fp32 cosine, bit-identical to br_cosine_rerank for row d (row_group_dev == NULL: row = doc, and n_rows must
 *           equal the index's n_docs), or to br_cosine_rerank_grouped for group d (row_group_dev as there, with the
 *           index's docs as the groups: n_groups = n_docs); a doc without rows has no cosine.  doc_inv_norm_dev from
 *           br_row_inv_norms; d a multiple of 8 and <= 1024, BR_ERR_UNSUPPORTED otherwise.
 *   Per query over the union: n_b = (s_b - min_b) / (max_b - min_b); n_c = ((double)s_c - min_c) / (max_c - min_c) over
 *   the members with a cosine, 0.0 for a doc without rows; a normalised value is 0.0 when max == min.  (1 - alpha) is
 *   formed once; every operation is one float64 rounding, no contraction.
 * out_bm25_dev double[nq, k] = s_b and out_cos_dev float[nq, k] = s_c of each returned doc (NaN: no rows; 0 pads); both
 * may be NULL.  The row_group layout is checked as in the grouped calls. */
int br_fuse_linear(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq, int32_t n_terms,
                   int dedup, const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_rows, int32_t d,
                   const int32_t* row_group_dev, const void* queries_bf16_dev, const int32_t* bm25_ids_dev, int32_t nb,
                   const int32_t* dense_ids_dev, int32_t nd, double alpha, int32_t k, int32_t* out_ids_dev,
                   double* out_scores_dev, double* out_bm25_dev, float* out_cos_dev, int32_t* out_counts_dev, void* stream);

/* Sentence -> document step of the sentence-level retrieval (team_run1.py:286-294): for every query walk its ranked
 * sentences sentence_ids_dev int64[nq, n] (best first, -1 = padding), map each to its parent doc through
 * sentence_to_doc_dev int32[n_sentences], keep the first occurrence of every doc and stop at k docs (k <= 32; the
 * reference uses 10).  out_docs_dev int64[nq, k], -1 pads.  Synchronises `stream`. */
int br_dedupe_first_docs(const int64_t* sentence_ids_dev, const int32_t* sentence_to_doc_dev, int64_t n_sentences,
                         int32_t nq, int32_t n, int32_t k, int64_t* out_docs_dev, void* stream);

/* Stream-ordered scratch of the handle-less entry points (cosine, text ingestion) comes from a private memory pool of the
 * library (one per device) that retains up to 8 GiB between calls; this returns all of it to the driver.  The process's
 * default memory pool is never touched. */
int br_trim_scratch(void);

/* Counters of the last br_topk_batch call on this handle (bench / tests): kernels launched,
 * queries served by the fused tiled path, by the dense path, and candidate rows re-scored. */
typedef struct br_query_stats {
    int64_t kernel_launches;
    int64_t queries_fused;
    int64_t queries_dense;
    int64_t candidates_rescored;
    int64_t postings_bytes;      /* algorithmic bytes: 8 * sum over queries of sum df (local shard) */
    int64_t score_launches;      /* launches of the scoring kernel (the dominant kernel) */
    double score_ms;             /* their summed device time (CUDA events on `stream`); 0 unless
                                    br_set_profiling(ix, 1) */
} br_query_stats;
int br_last_query_stats(const br_index* ix, br_query_stats* out);
/* Bracket every launch of the scoring kernel with CUDA events on the call's stream (bench.py's
 * live roofline measurement).  Off by default. */
int br_set_profiling(br_index* ix, int on);
/* Tuning / test switches.  name = "fused" (0 forces the dense path for every query; default 1), "fused_long" (0 sends
 * the queries the regular tiled pass cannot serve straight to the dense path instead of the long-query tiled pass;
 * default 1), "defer_pm" (MaxScore deferral budget of the tiled scorer in per mille of the threshold, 0-1000, 0 = off;
 * default 650).  Any other name: BR_ERR_INVALID. */
int br_set_option(br_index* ix, const char* name, int value);

/* ---------------------------------------------------------------------------------------------
 * Text ingestion: preprocessed text -> term ids (the step right before the index build).
 * Replaces `lang_tokenized_corpus = [text.split() for text in lang_texts]`
 * (bm25_ranking.ipynb:299), the first-seen vocabulary that the dict inserts of BM25.build create
 * (bm25_ranking.ipynb:180-186) and, with bigrams != 0, the 2-gram expansion
 * `tokens + ['_'.join(gram) for gram in ngrams(tokens, 2)]` (bm25_ranking.ipynb:105-107).
 *
 * text_dev is one UTF-8 buffer holding all documents back to back; doc_byte_off_dev int64[n_docs+1]
 * gives each document's byte range (the Arrow large_string layout).  Tokens are maximal runs of
 * characters for which Python's str.isspace() is false (str.split() semantics, Unicode whitespace
 * included); a token never crosses a document boundary.  Term ids are dense, in order of first
 * occurrence (document order; inside a document unigrams first, then bigrams), i.e. the insertion
 * order of the reference's dicts.  Terms are matched through a 64-bit hash and every token is
 * byte-compared with the first occurrence of its term: a hash collision is an error
 * (BR_ERR_UNSUPPORTED), never a silent merge.
 *
 * Call order: br_tokenize_count (fills doc_tok_off_dev int64[n_docs+1] = br_index_build's
 * doc_offsets, returns the token total) -> caller allocates token_ids_dev int32[n_tokens] ->
 * br_vocab_build (corpus: creates the vocabulary) or br_vocab_lookup (queries: ids under an
 * existing vocabulary, -1 = out of vocabulary, which the scoring kernels skip like
 * `if word not in self.idf: continue`, bm25_ranking.ipynb:195-196).  All three synchronise `stream`.
 * Limits per call: fewer than 2^31 tokens, documents shorter than 2 GiB (BR_ERR_UNSUPPORTED otherwise); scratch memory
 * is about 40 bytes per token, taken from the device's default stream-ordered pool. */
typedef struct br_vocab br_vocab;
int br_tokenize_count(const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs, int bigrams,
                      int64_t* doc_tok_off_dev, int64_t* n_tokens_host, void* stream);
int br_vocab_build(const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs, int bigrams,
                   const int64_t* doc_tok_off_dev, int64_t n_tokens, int32_t* token_ids_dev, void* stream,
                   br_vocab** out);
int br_vocab_lookup(const br_vocab* v, const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs,
                    int bigrams, const int64_t* doc_tok_off_dev, int64_t n_tokens, int32_t* token_ids_dev,
                    void* stream);
/* Grow a vocabulary with the tokens of new documents (call order as for br_vocab_build: br_tokenize_count first).
 * Writes the term id of every token to token_ids_dev.  A term already in v keeps its id.  New terms get ids
 * n_terms_old .. in order of first occurrence in the new text, which is the id br_vocab_build would give them over
 * old text + new text.  A 64-bit hash collision with an existing or another new term is BR_ERR_UNSUPPORTED.
 * On any error v is unchanged.  Synchronises `stream`. */
int br_vocab_extend(br_vocab* v, const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs, int bigrams,
                    const int64_t* doc_tok_off_dev, int64_t n_tokens, int32_t* token_ids_dev, void* stream);
int br_vocab_stats(const br_vocab* v, int64_t* n_terms, int64_t* pool_bytes);
/* Vocabulary strings: term t = pool[pool_off[t] .. pool_off[t+1]) (UTF-8).  Export for the Python
 * dict attributes (df / idf / inverted_index keys) and for pickling; import rebuilds the hash table. */
int br_vocab_export(const br_vocab* v, int64_t* pool_off_host, uint8_t* pool_host);
int br_vocab_import(const int64_t* pool_off_host, const uint8_t* pool_host, int64_t n_terms, void* stream,
                    br_vocab** out);
void br_vocab_destroy(br_vocab* v);

#ifdef __cplusplus
}
#endif
#endif /* BR_B200_H */
