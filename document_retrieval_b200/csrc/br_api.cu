// br_api.cu - C ABI (query side), error reporting, version.
#include "br_common.cuh"
#include "br_query.cuh"

namespace br {
static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
}  // namespace br

extern "C" {

const char* br_last_error(void) { return br::g_err.c_str(); }
const char* br_version(void) { return "br_b200 0.1 sm_100a"; }

int br_score_batch(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq, int dedup,
                   float* out_scores_dev, void* stream) {
    return br::score_batch(ix, q_terms_dev, q_offsets_dev, nq, dedup, out_scores_dev, (cudaStream_t)stream);
}

int br_topk_batch_filtered(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                           int32_t n_terms, int32_t k, int dedup, int positive_only, int32_t* out_ids_dev,
                           double* out_scores_dev, int32_t* out_counts_dev, const br_doc_filter* filter, void* stream) {
    BR_REQUIRE(out_ids_dev && out_scores_dev, BR_ERR_INVALID, "br_topk_batch: null pointer");
    return br::topk_batch(ix, q_terms_dev, q_offsets_dev, nq, n_terms, k, dedup, positive_only, out_ids_dev, out_scores_dev,
                          out_counts_dev, nullptr, filter, (cudaStream_t)stream);
}

int br_topk_batch(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq, int32_t n_terms,
                  int32_t k, int dedup, int positive_only, int32_t* out_ids_dev, double* out_scores_dev,
                  int32_t* out_counts_dev, void* stream) {
    return br_topk_batch_filtered(ix, q_terms_dev, q_offsets_dev, nq, n_terms, k, dedup, positive_only, out_ids_dev,
                                  out_scores_dev, out_counts_dev, nullptr, stream);
}

int br_topk_batch_records_filtered(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                                   int32_t n_terms, int32_t k, int dedup, int positive_only, br_record* out_records_dev,
                                   int32_t* out_counts_dev, const br_doc_filter* filter, void* stream) {
    BR_REQUIRE(out_records_dev, BR_ERR_INVALID, "br_topk_batch_records: null pointer");
    return br::topk_batch(ix, q_terms_dev, q_offsets_dev, nq, n_terms, k, dedup, positive_only, nullptr, nullptr,
                          out_counts_dev, out_records_dev, filter, (cudaStream_t)stream);
}

int br_topk_batch_records(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                          int32_t n_terms, int32_t k, int dedup, int positive_only, br_record* out_records_dev,
                          int32_t* out_counts_dev, void* stream) {
    return br_topk_batch_records_filtered(ix, q_terms_dev, q_offsets_dev, nq, n_terms, k, dedup, positive_only,
                                          out_records_dev, out_counts_dev, nullptr, stream);
}

int br_topk_merge_records(const br_record* records_dev, int32_t n_parts, int32_t nq, int32_t k, int64_t* out_ids_dev,
                          double* out_scores_dev, void* stream) {
    return br::topk_merge_records(records_dev, n_parts, nq, k, out_ids_dev, out_scores_dev, (cudaStream_t)stream);
}

int br_rescore_docs(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq, int dedup,
                    const int32_t* cand_ids_dev, const int64_t* cand_off_dev, double* out_scores_dev, void* stream) {
    return br::rescore_docs(ix, q_terms_dev, q_offsets_dev, nq, dedup, cand_ids_dev, cand_off_dev, out_scores_dev,
                            (cudaStream_t)stream);
}

int br_index_enable_tfidf(br_index* ix, void* stream) { return br::enable_tfidf(ix, (cudaStream_t)stream); }

int br_tfidf_cosine_topk(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq, int32_t k,
                         int32_t* out_ids_dev, double* out_scores_dev, int32_t* out_counts_dev, void* stream) {
    return br::tfidf_topk(ix, q_terms_dev, q_offsets_dev, nq, k, out_ids_dev, out_scores_dev, out_counts_dev,
                          (cudaStream_t)stream);
}

int br_rerank_v3_scores(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq,
                        const int32_t* cand_ids_dev, const int64_t* cand_off_dev, double* out_scores_dev, void* stream) {
    return br::rerank_v3(ix, q_terms_dev, q_offsets_dev, nq, cand_ids_dev, cand_off_dev, out_scores_dev, (cudaStream_t)stream);
}

int br_topk_merge(const int64_t* ids_dev, const double* scores_dev, int32_t n_parts, int32_t nq, int32_t k,
                  int64_t* out_ids_dev, double* out_scores_dev, void* stream) {
    return br::topk_merge(ids_dev, scores_dev, n_parts, nq, k, out_ids_dev, out_scores_dev, (cudaStream_t)stream);
}

int br_set_thr_exchange(br_index* ix, br_thr_exchange_fn fn, void* user, int rounds, int world) {
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_set_thr_exchange: null handle");
    BR_REQUIRE(!fn || (world >= 1 && world <= 16), BR_ERR_INVALID, "br_set_thr_exchange: world must be in [1, 16]");
    ix->thr_exchange_world = fn ? world : 1;
    ix->thr_exchange = fn;
    ix->thr_exchange_user = user;
    ix->thr_exchange_rounds = fn ? rounds : -1;
    return BR_OK;
}

int br_tile_launch_count(const br_index* ix, int32_t k) {
    if (!ix || !ix->finalized || k < 1 || k > BR_MAX_K) return 0;
    return br::fused_launch_count(ix, k);
}

int br_trim_scratch(void) {
    int dev = 0;
    BR_CUDA(cudaGetDevice(&dev));
    cudaMemPool_t pool = br::scratch_pool_slot(dev);
    if (pool) BR_CUDA(cudaMemPoolTrimTo(pool, 0));
    return BR_OK;
}

int br_last_query_stats(const br_index* ix, br_query_stats* out) {
    BR_REQUIRE(ix && out, BR_ERR_INVALID, "br_last_query_stats: null pointer");
    *out = ix->stats;
    return BR_OK;
}

int br_set_profiling(br_index* ix, int on) {
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_set_profiling: null handle");
    ix->profiling = on != 0;
    return BR_OK;
}

int br_set_option(br_index* ix, const char* name, int value) {
    BR_REQUIRE(ix && name, BR_ERR_INVALID, "br_set_option: null pointer");
    const std::string n(name);
    if (n == "fused") ix->allow_fused = value != 0;
    else if (n == "fused_long") ix->allow_fused_long = value != 0;
    else if (n == "defer_pm") {
        BR_REQUIRE(value >= 0 && value <= 1000, BR_ERR_INVALID, "br_set_option: defer_pm must be in [0, 1000]");
        ix->defer_pm = value;
    } else {
        br::set_error("br_set_option: unknown option " + n);
        return BR_ERR_INVALID;
    }
    return BR_OK;
}

}  // extern "C"
