// br_common.cuh - shared declarations of the br_b200 library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/br_b200.h"

namespace br {

// docs per skip-table sub-range = docs per warp of the tile kernel (2^kSubShift; why 2048: br_tile.cu)
constexpr int kSubShift = 11;

void set_error(const std::string& msg);

#define BR_CUDA(call)                                                                       \
    do {                                                                                    \
        cudaError_t _e = (call);                                                            \
        if (_e != cudaSuccess) {                                                            \
            br::set_error(std::string(#call) + ": " + cudaGetErrorString(_e) + " (" +       \
                          __FILE__ + ":" + std::to_string(__LINE__) + ")");                 \
            return BR_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

#define BR_TRY(call)                  \
    do {                              \
        int _s = (call);              \
        if (_s != BR_OK) return _s;   \
    } while (0)

#define BR_REQUIRE(cond, status, msg) \
    do {                              \
        if (!(cond)) {                \
            br::set_error(msg);       \
            return status;            \
        }                             \
    } while (0)

// One cudaMalloc allocation of T, freed with cudaFree by its owner: at the next alloc, at reset() or when it goes away.
// Converts to T* so that it reads like the raw device pointer it owns.
template <class T>
class DevArray {
  public:
    DevArray() = default;
    DevArray(DevArray&& o) noexcept : p_(o.p_) { o.p_ = nullptr; }
    DevArray& operator=(DevArray&& o) noexcept {
        if (this != &o) {
            reset();
            p_ = o.p_;
            o.p_ = nullptr;
        }
        return *this;
    }
    ~DevArray() { reset(); }
    // max(n, 1) elements; a failure names the caller's file and line
    int alloc(size_t n, const char* file = __builtin_FILE(), int line = __builtin_LINE()) {
        reset();
        const size_t bytes = sizeof(T) * std::max<size_t>(n, 1);
        const cudaError_t e = cudaMalloc(&p_, bytes);
        if (e == cudaSuccess) return BR_OK;
        p_ = nullptr;
        set_error("cudaMalloc(" + std::to_string(bytes) + " bytes): " + cudaGetErrorString(e) + " (" + file + ":" +
                  std::to_string(line) + ")");
        return BR_ERR_CUDA;
    }
    void reset() {
        if (p_) cudaFree(p_);
        p_ = nullptr;
    }
    T* get() const { return p_; }
    operator T*() const { return p_; }

  private:
    T* p_ = nullptr;
};

// Grow-only device workspace (never shrinks; freed with its owner).
struct DevBuf {
    DevArray<unsigned char> mem;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return BR_OK;
        cap = 0;
        const size_t want = bytes + bytes / 4 + 256;
        BR_TRY(mem.alloc(want));
        cap = want;
        return BR_OK;
    }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(mem.get()); }
};

// Stream-ordered scratch comes from a PRIVATE memory pool of the library, one per device: with a release threshold of 0
// every stream synchronisation would hand freed memory back to the driver and the next call pay for mapping it again
// (tens of ms for the larger buffers), so the pool keeps up to kPoolKeepBytes; anything above that is released at the
// next synchronisation.  The process's default pool (and with it the host application's own stream-ordered allocations)
// is left alone; br_trim_scratch() returns the retained memory on request.
constexpr uint64_t kPoolKeepBytes = 8ull << 30;
inline cudaMemPool_t& scratch_pool_slot(int dev) {
    static cudaMemPool_t pools[64] = {};
    return pools[dev & 63];
}
inline int scratch_pool(cudaMemPool_t* out) {
    int dev = 0;
    BR_CUDA(cudaGetDevice(&dev));
    cudaMemPool_t& pool = scratch_pool_slot(dev);
    if (!pool) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        BR_CUDA(cudaMemPoolCreate(&pool, &props));
        uint64_t keep = kPoolKeepBytes;
        BR_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    *out = pool;
    return BR_OK;
}
inline int scratch_alloc(void** p, size_t bytes, cudaStream_t st) {
    cudaMemPool_t pool;
    BR_TRY(scratch_pool(&pool));
    BR_CUDA(cudaMallocFromPoolAsync(p, bytes ? bytes : 1, pool, st));
    return BR_OK;
}
// The stream-ordered temporaries of one call: every alloc comes from the scratch pool and is freed on the same stream
// (cudaFreeAsync) when the scope ends, whichever way the call returns.
class StreamScratch {
  public:
    explicit StreamScratch(cudaStream_t st) : st_(st) {}
    StreamScratch(const StreamScratch&) = delete;
    StreamScratch& operator=(const StreamScratch&) = delete;
    ~StreamScratch() {
        for (void* p : ptrs_) cudaFreeAsync(p, st_);
    }
    template <class T>
    int alloc(T** out, size_t n) {   // max(n, 1) elements
        void* p = nullptr;
        BR_TRY(scratch_alloc(&p, sizeof(T) * std::max<size_t>(n, 1), st_));
        ptrs_.push_back(p);
        *out = static_cast<T*>(p);
        return BR_OK;
    }

  private:
    cudaStream_t st_;
    std::vector<void*> ptrs_;
};

constexpr int kNumSMs = 148;          // B200
constexpr float kBandRel = 1e-5f;     // fp32 candidate band kept below the k-th fp32 score (see DESIGN.md)

// Per-query doc filter of a batch (br_doc_filter after validation): query q may return local doc d iff row[q] < 0 or bit
// (d & 31) of word (d >> 5) of bitmap row row[q] is set.  row[] is indexed like the kernel's query index (a sub-batch gets
// its own remapped copy) and holds only values in [-1, n_rows).
struct DocFilter {
    const uint32_t* bits;
    int64_t words;
    const int32_t* row;
#ifdef __CUDACC__
    __device__ __forceinline__ const uint32_t* row_of(int q) const {
        const int32_t r = row[q];
        return r < 0 ? nullptr : bits + (int64_t)r * words;
    }
#endif
};
#ifdef __CUDACC__
// fr: the query's bitmap row (nullptr: unfiltered); doc < n_docs
__device__ __forceinline__ bool doc_allowed(const uint32_t* fr, uint32_t doc) {
    return !fr || ((__ldg(fr + (doc >> 5)) >> (doc & 31)) & 1u) != 0u;
}
#endif

}  // namespace br

// One posting: doc id + precomputed fp32 BM25 weight, 8 bytes, read as one 64-bit word
// (two postings per 128-bit load).
struct __align__(8) br_posting {
    uint32_t doc;
    float w;
};

struct br_index {
    int device = 0;
    int64_t n_docs = 0, doc_base = 0, nnz = 0, sum_dl = 0;
    int32_t vocab = 0;
    bool finalized = false;
    int variant = 0;
    double k1 = 1.5, b = 0.75, n_stat = 0, sum_dl_stat = 0, avgdl = 0;

    // CSR by term (device)
    br::DevArray<int64_t> row_ptr;     // [V+1]
    br::DevArray<br_posting> post;     // [nnz]   doc ids ascending inside a term
    br::DevArray<br_posting> post_cos; // [nnz]   optional TF-IDF cosine weights tf*idf^2/||d|| (br_index_enable_tfidf)
    br::DevArray<double> cos_inv_norm; // [N]     1/||d|| of the doc's float32 tf*idf vector, float64 (with post_cos)
    br::DevArray<uint16_t> tf;         // [nnz]   raw term frequency (for the float64 re-score)
    br::DevArray<uint32_t> dl;         // [N]
    br::DevArray<uint32_t> df;         // [V]     shard-local document frequency
    br::DevArray<double> idf;          // [V]     statistics in force (NaN where df_stat == 0)
    br::DevArray<float> ub;            // [V]     largest posting weight of the term on this shard (0 when none / negative):
                                       //         the per-term score upper bound of the tiled scorer's MaxScore deferral
    br::DevArray<float> amax;          // [V]     largest |posting weight| of the term on this shard; okapi_no_plus1 only
                                       //         (null otherwise): the fp32 error bound of a query with mixed signs

    // hot-term skip tables for the tiled scorer: term t is "hot" when hot_slot[t] >= 0; then
    // skip[hot_slot[t] * (n_sub+1) + j] = offset (relative to row_ptr[t]) of the first posting
    // with doc >= j << sub_shift.
    int sub_shift = 0;
    int32_t n_sub = 0, n_hot = 0;
    uint32_t hot_min = 0;           // smallest df with a skip table
    br::DevArray<int32_t> hot_slot;    // [V]
    br::DevArray<uint32_t> skip;       // [n_hot, n_sub+1]
    // dense rows: w[row][doc] as plain fp32 rows (0 where the doc lacks the term), most frequent term first.
    // Rows [0, n_srows) - terms present in >= ~20% of the docs - are STREAMED by the tiled scorer (accumulators are
    // initialised from them instead of walking their postings); all n_rows rows (terms with df >= N/64) serve as
    // LOOK-UP tables: a term the scorer has deferred (MaxScore) is added to a candidate doc with one 4-byte load.
    br::DevArray<float> dense_rows;    // [n_rows, n_pad]
    br::DevArray<int16_t> row_slot;    // [V] row index or -1
    int32_t n_rows = 0, n_srows = 0;
    int64_t n_pad = 0;
    br::DevArray<int8_t> sig_bit;      // [V] rank (0 = largest df) among the 32 most frequent terms, -1 otherwise

    // host mirrors
    std::vector<uint32_t> h_df;     // shard-local
    std::vector<int64_t> h_df_stat; // statistics in force
    std::vector<double> h_idf;

    // query-time scratch
    br::DevBuf ws_prep, ws_dense, ws_sel, ws_cand, ws_misc, ws_tile, ws_sort, ws_cold, ws_rec;
    br::DevBuf ws_filt;             // filtered batches: validated filter rows of the batch and of its redo sub-batch
    br_query_stats stats{};

    bool allow_fused = true, allow_fused_long = true;
    // doc-sharded callers: callback that max-reduces thr[Q] over the shards (br_set_thr_exchange), user pointer, and the
    // number of tile launches after which it is called (plus once after seeding); rounds < 0: off
    br_thr_exchange_fn thr_exchange = nullptr;
    void* thr_exchange_user = nullptr;
    int thr_exchange_rounds = -1;
    int thr_exchange_world = 1;
    int defer_pm = 650;             // MaxScore deferral budget of the tiled scorer, per mille of the threshold (0 = off)

    // optional event timing of the scoring kernel
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;   // pairs (start, stop)
    size_t ev_used = 0;
    ~br_index() {
        for (cudaEvent_t e : ev_pool) cudaEventDestroy(e);
    }
    void prof_begin(cudaStream_t st) {
        if (!profiling) return;
        if (ev_used + 2 > ev_pool.size()) {
            cudaEvent_t a, b;
            cudaEventCreate(&a); cudaEventCreate(&b);
            ev_pool.push_back(a); ev_pool.push_back(b);
        }
        cudaEventRecord(ev_pool[ev_used], st);
    }
    void prof_end(cudaStream_t st) {
        stats.score_launches += 1;
        if (!profiling) return;
        cudaEventRecord(ev_pool[ev_used + 1], st);
        ev_used += 2;
    }
    void prof_collect() {   // call after the stream is synchronised
        for (size_t i = 0; i + 1 < ev_used; i += 2) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, ev_pool[i], ev_pool[i + 1]) == cudaSuccess) stats.score_ms += ms;
        }
        ev_used = 0;
    }
};

namespace br {
// br_build.cu
int index_build(const int32_t* token_ids, const int64_t* doc_offsets, int64_t n_docs, int32_t vocab,
                int64_t doc_base, cudaStream_t st, br_index** out);
int index_finalize(br_index* ix, double k1, double b, int variant, double n_stat, double sum_dl_stat,
                   const int64_t* df_stat_host, cudaStream_t st);
int index_import(const int64_t* row_ptr, const int32_t* doc, const int32_t* tf, const int32_t* dl,
                 int64_t n_docs, int32_t vocab, int64_t doc_base, cudaStream_t st, br_index** out);
int index_import_dev(const int64_t* row_ptr, const int32_t* doc, const uint16_t* tf, const int32_t* dl, int64_t n_docs,
                     int32_t vocab, int64_t nnz, int64_t doc_base, cudaStream_t st, br_index** out);
int index_append(br_index* ix, const int32_t* token_ids, const int64_t* doc_offsets, int64_t n_docs, int32_t vocab,
                 cudaStream_t st);
int index_remove(br_index* ix, const uint8_t* remove, cudaStream_t st);
void index_free(br_index* ix);
// br_query.cu
int score_batch(br_index* ix, const int32_t* q_terms, const int32_t* q_offsets, int32_t nq, int dedup,
                float* out_scores, cudaStream_t st);
int topk_batch(br_index* ix, const int32_t* q_terms, const int32_t* q_offsets, int32_t nq, int32_t n_terms, int32_t k,
               int dedup, int positive_only, int32_t* out_ids, double* out_scores, int32_t* out_counts,
               br_record* out_recs, const br_doc_filter* filter, cudaStream_t st);
int rescore_docs(br_index* ix, const int32_t* q_terms, const int32_t* q_offsets, int32_t nq, int dedup,
                 const int32_t* cand_ids, const int64_t* cand_off, double* out_scores, cudaStream_t st);
int enable_tfidf(br_index* ix, cudaStream_t st);
int tfidf_topk(br_index* ix, const int32_t* q_terms, const int32_t* q_offsets, int32_t nq, int32_t k, int32_t* out_ids,
               double* out_scores, int32_t* out_counts, cudaStream_t st);
int rerank_v3(br_index* ix, const int32_t* q_terms, const int32_t* q_offsets, int32_t nq, const int32_t* cand_ids,
              const int64_t* cand_off, double* out_scores, cudaStream_t st);
int topk_merge(const int64_t* ids, const double* scores, int32_t n_parts, int32_t nq, int32_t k,
               int64_t* out_ids, double* out_scores, cudaStream_t st);
int topk_merge_records(const br_record* recs, int32_t n_parts, int32_t nq, int32_t k, int64_t* out_ids,
                       double* out_scores, cudaStream_t st);
}  // namespace br
