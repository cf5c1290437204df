// br_query.cuh - declarations shared by br_query.cu (dense path, re-score, final select, doc filters) with
// br_tile.cu (fused tiled path), br_cosine.cu (dense cosine) and br_hybrid.cu (BM25 + dense fusion).
#pragma once
#include "br_common.cuh"

namespace br {

struct PrepView {
    int32_t* u_terms;   // [T]  per query segment: unique valid terms ascending
    int32_t* u_mult;    // [T]  multiplicity (1 when dedup)
    int64_t* u_cum;     // [T]  exclusive prefix of df over the unique terms
    int32_t* u_cnt;     // [nq]
    int32_t* o_terms;   // [T]  valid terms in query order (duplicates kept)
    int32_t* o_cnt;     // [nq]
    int64_t* P;         // [nq] total postings of the unique terms
    uint32_t* n_chunks; // [nq]
    int32_t* tmp;       // [T]
    uint32_t* sig;      // [nq] bit (31 - r) set when the query contains the r-th most frequent term
    float* slack;       // [nq] > 0 for a query with a term of negative idf: twice the bound on |fp32 sum - float64
                        //      score| of any doc, (2n + 6) 2^-24 sum_t mult_t amax_t over its n distinct terms; else 0
    int32_t t_cap;      // term slots the scratch arrays hold (caller's n_terms)
    int32_t* bad;       // [1] set when q_offsets runs past t_cap
};


// The query preparation of br_topk_batch (k_prep_queries into ix->ws_prep); n_terms < 0: read q_offsets[nq] back.
int prep_queries(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int dedup, cudaStream_t st,
                 PrepView* pv, int64_t** chunk_start, int32_t n_terms = -1);
// The float64 formula of an exact re-score: BM25 (br_topk_batch, br_rescore_docs), TF-IDF cosine (br_tfidf_cosine_topk),
// V3 re-rank (br_rerank_v3_scores).  An empty candidate slot (id -1) gets 0.0.
enum class Formula { BM25, COS, V3 };
// Candidates of query q in [cand_off[q], cand_off[q+1]), q in [q_begin, q_begin + nq); total: their number, -1 when
// only the device knows it.
int launch_rescore(br_index* ix, Formula f, const int32_t* q_off, const PrepView& pv, int dedup, const int64_t* cand_off,
                   int32_t q_begin, int32_t nq, const int32_t* cand, double* cand_score, int64_t total, cudaStream_t st);
// Candidates of query q in the fixed-stride region [q * stride, (q+1) * stride), of which the first cnt[q] are live.
int launch_rescore_heads(br_index* ix, Formula f, const int32_t* q_off, const PrepView& pv, int dedup, int32_t nq,
                         int32_t stride, const int32_t* cnt, const int32_t* cand, double* cand_score, cudaStream_t st);
// cand_off == NULL: query q's candidates are [q * fixed_cnt, (q + 1) * fixed_cnt)
int launch_final_select(const int32_t* cand, const double* cand_score, const int64_t* cand_off, int32_t q_begin,
                        int32_t nq, int32_t k, int positive_only, int32_t* out_ids, double* out_scores,
                        int32_t* out_counts, cudaStream_t st, const int32_t* cnt_hint = nullptr, int32_t fixed_cnt = 0);
// The checks of a br_doc_filter argument (NULL: unfiltered, nothing to check) whose bitmap covers n_ids ids, named `ids`
// ("n_docs", "n_groups") in the message of the call `fn`.
int check_doc_filter(const br_doc_filter* filter, int64_t n_ids, const char* ids, const std::string& fn);
// Filter rows of a batch (br_doc_filter::query_row_dev, NULL = row 0 for every query), validated on the device: a value
// outside [-1, n_rows) sets *bad and becomes -1.
__global__ void k_filter_rows(const int32_t* __restrict__ in, int32_t nq, int32_t n_rows, int32_t* __restrict__ out,
                              int32_t* __restrict__ bad);
bool fused_supported(const br_index* ix, int32_t k, int32_t nq, bool cos = false);
int fused_launch_count(const br_index* ix, int32_t k);
int topk_fused(br_index* ix, const int32_t* q_off, const PrepView& pv, int32_t nq, int32_t k, int dedup,
               int positive_only, int32_t* out_ids, double* out_scores, int32_t* out_counts, cudaStream_t st,
               std::vector<int32_t>* h_flags, bool long_pass = false, const br_posting* post_table = nullptr,
               const DocFilter* filt = nullptr);

// br_cosine.cu: the gather kernels of br_cosine_rerank / br_cosine_rerank_grouped over fixed-stride candidate lists
// cand[q, 0..c) (-1 = empty slot), for callers that need the per-candidate cosines rather than a selection.
int row_inv_norms(const void* emb, int64_t n, int32_t d, float* out, cudaStream_t st);
// out[q, c] fp32 cosines (-inf for an empty slot); bad (may be NULL) is set when an id is outside [-1, n_docs).  d <= 1024.
int launch_cos_gather(const void* docs, const float* inv_nd, int64_t n_docs, int32_t d, const void* queries,
                      const float* inv_nq, int32_t nq, const int32_t* cand, int32_t c, float* out, int32_t* bad,
                      cudaStream_t st);
// Checks the row_group layout (failing the call `fn`), then per candidate: out_ids = its group, -1 for an empty slot, a
// group without rows or an id outside [-1, n_groups) (which sets *bad); out_s64 = the group's best cosine, widened
// (0.0 without rows).  d <= 1024.
int launch_cos_gather_grouped(const void* docs, const float* inv_nd, int64_t n_rows, int32_t d, const int32_t* row_group,
                              int32_t n_groups, const void* queries, const float* inv_nq, int32_t nq, const int32_t* cand,
                              int32_t c, int32_t* out_ids, double* out_s64, int32_t* bad, const std::string& fn,
                              cudaStream_t st);

}  // namespace br
