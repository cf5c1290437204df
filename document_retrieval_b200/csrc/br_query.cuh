// br_query.cuh - declarations shared by br_query.cu (dense path, re-score, final select, doc filters) with
// br_tile.cu (fused tiled path) and br_cosine.cu (dense cosine).
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
    int32_t t_cap;      // term slots the scratch arrays hold (caller's n_terms)
    int32_t* bad;       // [1] set when q_offsets runs past t_cap
};


int launch_rescore(br_index* ix, const int32_t* q_off, const PrepView& pv, int dedup, const int64_t* cand_off,
                   int32_t q_begin, int32_t nq, const int32_t* cand, double* cand_score, int64_t total, cudaStream_t st);
int launch_rescore_heads(br_index* ix, const int32_t* q_off, const PrepView& pv, int dedup, int32_t nq, int32_t stride,
                         const int32_t* cnt, const int32_t* cand, double* cand_score, cudaStream_t st, bool cos = false);
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

}  // namespace br
