// br_ingest.cu - text -> term ids on the GPU (SURVEY 8f rank 2: the step right before the hot path).
//
// Replaces, for whole corpora at once,
//   lang_tokenized_corpus = [text.split() for text in lang_texts]            bm25_ranking.ipynb:299
//   the per-token dict inserts of BM25.build (first-seen vocabulary order)    bm25_ranking.ipynb:180-186
//   tokens + ['_'.join(gram) for gram in ngrams(tokens, 2)]                   bm25_ranking.ipynb:105-107
// Input is an Arrow-style UTF-8 buffer (all documents concatenated, int64 byte offsets).
//
//   k_tok_count   warp per document: token starts by str.split() rules (Unicode whitespace) -> tokens per doc
//   k_exscan      -> doc_tok_off
//   k_tok_emit    warp per document: (start, length[, bigram flag]) of every token, unigrams first then bigrams
//   k_tok_hash    thread per token: 64-bit hash of the token's canonical bytes ("a_b" for a bigram)
//   CUB radix sort of (hash, token index)            [library plumbing, like the index build]
//   k_head_count / k_head_emit   runs of equal hashes -> distinct terms, first occurrence of each
//   CUB radix sort of (first occurrence, run)  -> term id = rank in first-seen order (dict insertion order)
//   k_assign      token -> term id, every token byte-compared with its term's first occurrence: a 64-bit hash
//                 collision is reported as an error instead of silently merging two terms
//   k_pool_len / k_pool_fill     vocabulary strings into one byte pool (-> Python `terms`, query-time verification)
//   k_lookup      query tokens: binary search in the sorted hash table + byte compare -> term id or -1 (OOV)
// Extension (br_vocab_extend): the new text's own vocabulary (the pipeline above), then
//   k_extend_find its terms looked up in the existing table (hash + byte compare), k_exscan numbers the new ones
//   k_extend_map  local id -> global id; k_remap the new tokens; k_extend_pool appends the new strings; the new
//                 (hash, id) pairs are sorted into the table together with the old ones
#include <memory>

#include <cub/cub.cuh>

#include "br_kernels.cuh"

struct br_vocab {
    int device = 0;
    int64_t n_terms = 0, pool_bytes = 0;
    br::DevArray<uint64_t> hash_sorted;   // [V] ascending
    br::DevArray<int32_t> term_sorted;    // [V] term id of hash_sorted[i]
    br::DevArray<int64_t> pool_off;       // [V+1]
    br::DevArray<uint8_t> pool;           // [pool_bytes]
};

namespace br {
namespace {

constexpr uint32_t kBigram = 0x80000000u;
constexpr int kTile = 1024;   // sorted positions per CTA in the run-length kernels

// length in bytes of the whitespace character that starts at p (0 if none): the characters for which Python's
// str.isspace() holds, i.e. what str.split() without arguments splits on.
__device__ __forceinline__ int ws_char(const uint8_t* __restrict__ t, int64_t p, int64_t hi) {
    const uint8_t c = t[p];
    if (c < 0x80) return (c == 0x20 || (c >= 0x09 && c <= 0x0d) || (c >= 0x1c && c <= 0x1f)) ? 1 : 0;
    if (c == 0xc2) {   // U+0085, U+00A0
        if (p + 1 < hi) {
            const uint8_t d = t[p + 1];
            if (d == 0x85 || d == 0xa0) return 2;
        }
        return 0;
    }
    if (c < 0xe1 || c > 0xe3 || p + 2 >= hi) return 0;
    const uint8_t d = t[p + 1], e = t[p + 2];
    if (c == 0xe1) return (d == 0x9a && e == 0x80) ? 3 : 0;   // U+1680
    if (c == 0xe2) {
        // U+2000-200A, U+2028, U+2029, U+202F | U+205F
        if (d == 0x80) return ((e >= 0x80 && e <= 0x8a) || e == 0xa8 || e == 0xa9 || e == 0xaf) ? 3 : 0;
        if (d == 0x81) return e == 0x9f ? 3 : 0;
        return 0;
    }
    return (d == 0x80 && e == 0x80) ? 3 : 0;   // U+3000
}

// is byte p part of a whitespace character?  [lo, hi) starts on a character boundary.
__device__ __forceinline__ bool ws_byte(const uint8_t* __restrict__ t, int64_t p, int64_t lo, int64_t hi) {
    const uint8_t c = t[p];
    if (c < 0x80) return c == 0x20 || (c >= 0x09 && c <= 0x0d) || (c >= 0x1c && c <= 0x1f);
    int64_t s = p;
    while (s > lo && (t[s] & 0xc0) == 0x80 && p - s < 3) --s;
    return ws_char(t, s, hi) > (int)(p - s);
}

// One pass of a warp over document [lo, hi): calls on_start(rank, p) / on_end(rank, p) for every token in order
// and returns the number of tokens.  Position hi is processed as a virtual whitespace byte so that a token running
// to the end of the document is closed there (documents are not separated by anything in the buffer).
template <class FS, class FE>
__device__ __forceinline__ uint32_t warp_scan_doc(const uint8_t* __restrict__ t, int64_t lo, int64_t hi, int lane,
                                                  FS on_start, FE on_end) {
    uint32_t n_start = 0, n_end = 0;
    bool carry = true;   // "previous byte is whitespace" for lane 0
    for (int64_t base = lo; base <= hi; base += 32) {
        const int64_t p = base + lane;
        const bool w = p < hi ? ws_byte(t, p, lo, hi) : true;
        bool prev = __shfl_up_sync(0xffffffffu, (int)w, 1) != 0;
        if (lane == 0) prev = carry;
        carry = __shfl_sync(0xffffffffu, (int)w, 31) != 0;
        const bool is_start = !w && prev && p < hi;
        const bool is_end = w && !prev && p <= hi;
        const uint32_t ms = __ballot_sync(0xffffffffu, is_start), me = __ballot_sync(0xffffffffu, is_end);
        const uint32_t below = (1u << lane) - 1u;
        if (is_start) on_start(n_start + __popc(ms & below), p);
        if (is_end) on_end(n_end + __popc(me & below), p);
        n_start += __popc(ms);
        n_end += __popc(me);
    }
    return n_start;
}

__global__ void __launch_bounds__(256) k_tok_count(const uint8_t* __restrict__ text, const int64_t* __restrict__ doc_off,
                                                   int64_t n_docs, int bigrams, uint32_t* __restrict__ counts,
                                                   int* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t d = warp0; d < n_docs; d += nwarps) {
        const int64_t lo = doc_off[d], hi = doc_off[d + 1];
        uint32_t n = 0;
        if (hi < lo) {
            if (lane == 0) atomicOr(bad, 2);
        } else if (hi - lo >= (int64_t)kBigram) {
            if (lane == 0) atomicOr(bad, 4);
        } else {
            n = warp_scan_doc(text, lo, hi, lane, [](uint32_t, int64_t) {}, [](uint32_t, int64_t) {});
            if (bigrams && n >= 2) n += n - 1;
        }
        if (lane == 0) counts[d] = n;
    }
}

__global__ void __launch_bounds__(256) k_tok_emit(const uint8_t* __restrict__ text, const int64_t* __restrict__ doc_off,
                                                  const int64_t* __restrict__ doc_tok_off, int64_t n_docs, int bigrams,
                                                  int64_t* __restrict__ tok_start, uint32_t* __restrict__ tok_len) {
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t d = warp0; d < n_docs; d += nwarps) {
        const int64_t lo = doc_off[d], hi = doc_off[d + 1];
        const int64_t o = doc_tok_off[d];
        const int64_t total = doc_tok_off[d + 1] - o;
        if (hi <= lo || total == 0) continue;
        // unigrams of this doc: total = n, or 2n-1 with bigrams and n >= 2
        const int64_t n = (bigrams && total >= 3) ? (total + 1) / 2 : total;
        int64_t* ts = tok_start + o;
        uint32_t* tl = tok_len + o;
        // pass: starts, and the low 32 bits of the (exclusive) ends - docs are < 2^31 bytes, so the length is
        // the modular difference
        warp_scan_doc(text, lo, hi, lane, [&](uint32_t r, int64_t p) { ts[r] = p; },
                      [&](uint32_t r, int64_t p) { tl[r] = (uint32_t)p; });
        __syncwarp();
        for (int64_t r = lane; r < n; r += 32) tl[r] = tl[r] - (uint32_t)ts[r];
        __syncwarp();
        if (bigrams && n >= 2) {
            for (int64_t r = lane; r < n - 1; r += 32) {
                const int64_t s = ts[r];
                ts[n + r] = s;
                tl[n + r] = (uint32_t)(ts[r + 1] + tl[r + 1] - s) | kBigram;   // span of both tokens
            }
        }
        __syncwarp();
    }
}

// Canonical bytes of a token: its own bytes, or for a bigram "first_second" read from the span of both tokens.
struct Canon {
    const uint8_t* t;
    int64_t p, lo, end;
    int phase;   // 1 = inside the first token of a bigram
    __device__ Canon(const uint8_t* t_, int64_t start, uint32_t len)
        : t(t_), p(start), lo(start), end(start + (int64_t)(len & ~kBigram)), phase((len & kBigram) ? 1 : 0) {}
    __device__ __forceinline__ int next() {
        if (phase == 1) {
            if (!ws_byte(t, p, lo, end)) return t[p++];
            phase = 0;
            while (p < end && ws_byte(t, p, lo, end)) ++p;
            return '_';
        }
        return p < end ? (int)t[p++] : -1;
    }
};

__device__ __forceinline__ uint64_t fmix64(uint64_t k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL;
    k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL;
    k ^= k >> 33;
    return k;
}

__device__ __forceinline__ uint64_t canon_hash(Canon c) {
    uint64_t h = 0xcbf29ce484222325ULL;   // FNV-1a over the bytes, then a murmur finaliser
    int b;
    while ((b = c.next()) >= 0) h = (h ^ (uint64_t)b) * 0x100000001b3ULL;
    return fmix64(h);
}

__device__ __forceinline__ bool canon_equal(Canon a, Canon b) {
    for (;;) {
        const int x = a.next(), y = b.next();
        if (x != y) return false;
        if (x < 0) return true;
    }
}

__global__ void __launch_bounds__(256) k_tok_hash(const uint8_t* __restrict__ text, const int64_t* __restrict__ tok_start,
                                                  const uint32_t* __restrict__ tok_len, int64_t n_tok,
                                                  uint64_t* __restrict__ hash, uint32_t* __restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tok) return;
    hash[i] = canon_hash(Canon(text, tok_start[i], tok_len[i]));
    if (idx) idx[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(kTile) k_head_count(const uint64_t* __restrict__ key, int64_t n,
                                                      uint32_t* __restrict__ block_counts) {
    const int64_t i = (int64_t)blockIdx.x * kTile + threadIdx.x;
    const int flag = i < n && (i == 0 || key[i] != key[i - 1]);
    const int c = __syncthreads_count(flag);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = (uint32_t)c;
}

__global__ void __launch_bounds__(kTile) k_head_emit(const uint64_t* __restrict__ key, const uint32_t* __restrict__ val,
                                                     int64_t n, const int64_t* __restrict__ block_off,
                                                     uint64_t* __restrict__ hash_u, uint32_t* __restrict__ first_tok,
                                                     uint32_t* __restrict__ run_id) {
    const int64_t i = (int64_t)blockIdx.x * kTile + threadIdx.x;
    const uint32_t flag = i < n && (i == 0 || key[i] != key[i - 1]);
    uint32_t total;
    const uint32_t ex = block_excl_scan(flag, &total);
    if (flag) {
        const int64_t u = block_off[blockIdx.x] + ex;
        hash_u[u] = key[i];
        first_tok[u] = val[i];
        run_id[u] = (uint32_t)u;
    }
}

__global__ void k_rank_scatter(const uint32_t* __restrict__ run_sorted, int64_t n_terms, int32_t* __restrict__ term_of_run) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n_terms) term_of_run[run_sorted[r]] = (int32_t)r;
}

__global__ void __launch_bounds__(kTile) k_assign(const uint8_t* __restrict__ text, const int64_t* __restrict__ tok_start,
                                                  const uint32_t* __restrict__ tok_len, const uint64_t* __restrict__ key,
                                                  const uint32_t* __restrict__ val, int64_t n,
                                                  const int64_t* __restrict__ block_off,
                                                  const uint32_t* __restrict__ first_tok,
                                                  const int32_t* __restrict__ term_of_run, int32_t* __restrict__ token_ids,
                                                  int* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * kTile + threadIdx.x;
    const uint32_t flag = i < n && (i == 0 || key[i] != key[i - 1]);
    uint32_t total;
    const uint32_t ex = block_excl_scan(flag, &total);
    if (i >= n) return;
    // run of this position: heads before it in the CTA, minus one unless it is a head itself; a CTA that starts
    // inside a run continues the last run of the CTAs before it
    const int64_t u = block_off[blockIdx.x] + ex + flag - 1;
    const uint32_t tok = val[i];
    token_ids[tok] = term_of_run[u];
    if (!flag) {
        const uint32_t f = first_tok[u];
        if (!canon_equal(Canon(text, tok_start[tok], tok_len[tok]), Canon(text, tok_start[f], tok_len[f])))
            atomicOr(bad, 8);   // two different strings with the same 64-bit hash
    }
}

__global__ void k_pool_len(const uint8_t* __restrict__ text, const int64_t* __restrict__ tok_start,
                           const uint32_t* __restrict__ tok_len, const uint32_t* __restrict__ first_by_rank,
                           int64_t n_terms, uint32_t* __restrict__ clen) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_terms) return;
    const uint32_t tok = first_by_rank[r];
    const uint32_t len = tok_len[tok];
    if (!(len & kBigram)) { clen[r] = len; return; }
    Canon c(text, tok_start[tok], len);
    uint32_t m = 0;
    while (c.next() >= 0) ++m;
    clen[r] = m;
}

__global__ void k_pool_fill(const uint8_t* __restrict__ text, const int64_t* __restrict__ tok_start,
                            const uint32_t* __restrict__ tok_len, const uint32_t* __restrict__ first_by_rank,
                            int64_t n_terms, const int64_t* __restrict__ pool_off, uint8_t* __restrict__ pool) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_terms) return;
    const uint32_t tok = first_by_rank[r];
    Canon c(text, tok_start[tok], tok_len[tok]);
    uint8_t* o = pool + pool_off[r];
    int b;
    while ((b = c.next()) >= 0) *o++ = (uint8_t)b;
}

__global__ void k_pool_hash(const uint8_t* __restrict__ pool, const int64_t* __restrict__ pool_off, int64_t n_terms,
                            uint64_t* __restrict__ hash, uint32_t* __restrict__ term) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_terms) return;
    const int64_t s = pool_off[r];
    hash[r] = canon_hash(Canon(pool, s, (uint32_t)(pool_off[r + 1] - s)));
    term[r] = (uint32_t)r;
}

__global__ void k_dup_check(const uint64_t* __restrict__ key, int64_t n, int* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > 0 && i < n && key[i] == key[i - 1]) atomicOr(bad, 8);
}

__global__ void k_u32_to_i32(const uint32_t* __restrict__ in, int64_t n, int32_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int32_t)in[i];
}

__global__ void __launch_bounds__(256) k_lookup(const uint8_t* __restrict__ text, const int64_t* __restrict__ tok_start,
                                                const uint32_t* __restrict__ tok_len, int64_t n_tok,
                                                const uint64_t* __restrict__ hash_sorted,
                                                const int32_t* __restrict__ term_sorted, int64_t n_terms,
                                                const int64_t* __restrict__ pool_off, const uint8_t* __restrict__ pool,
                                                int32_t* __restrict__ token_ids) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_tok) return;
    const Canon c(text, tok_start[i], tok_len[i]);
    const uint64_t h = canon_hash(c);
    int64_t lo = 0, hi = n_terms;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (hash_sorted[mid] < h) lo = mid + 1; else hi = mid;
    }
    int32_t term = -1;   // out of vocabulary: skipped by the scoring kernels like `if word not in self.idf: continue`
    if (lo < n_terms && hash_sorted[lo] == h) {
        const int32_t t = term_sorted[lo];
        const int64_t s = pool_off[t];
        if (canon_equal(c, Canon(pool, s, (uint32_t)(pool_off[t + 1] - s)))) term = t;
    }
    token_ids[i] = term;
}

// Vocabulary extension, thread per entry i of the new text's own (local) hash table: is its term in v?  A hash hit is
// byte-compared like k_lookup; a hit with other bytes is a collision.  By local id r: known[r] = the term id in v or -1,
// is_new[r] = known[r] < 0, hash_of[r] = the term's hash.
__global__ void k_extend_find(const uint64_t* __restrict__ loc_hash, const int32_t* __restrict__ loc_term, int64_t n_loc,
                              const int64_t* __restrict__ loc_pool_off, const uint8_t* __restrict__ loc_pool,
                              const uint64_t* __restrict__ hash_sorted, const int32_t* __restrict__ term_sorted,
                              int64_t n_terms, const int64_t* __restrict__ pool_off, const uint8_t* __restrict__ pool,
                              int32_t* __restrict__ known, uint32_t* __restrict__ is_new, uint64_t* __restrict__ hash_of,
                              int* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_loc) return;
    const uint64_t h = loc_hash[i];
    const int32_t r = loc_term[i];
    int64_t lo = 0, hi = n_terms;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (hash_sorted[mid] < h) lo = mid + 1; else hi = mid;
    }
    int32_t term = -1;
    if (lo < n_terms && hash_sorted[lo] == h) {
        const int32_t t = term_sorted[lo];
        const int64_t s = pool_off[t], ls = loc_pool_off[r];
        if (canon_equal(Canon(loc_pool, ls, (uint32_t)(loc_pool_off[r + 1] - ls)), Canon(pool, s, (uint32_t)(pool_off[t + 1] - s))))
            term = t;
        else
            atomicOr(bad, 8);
    }
    known[r] = term;
    is_new[r] = term < 0 ? 1u : 0u;
    hash_of[r] = h;
}

// By local id r: map[r] = the global term id (a new term's is n_terms + its rank among the new terms in local, i.e.
// first-occurrence, order); a new term also gets its slot in the appended hash entries and its string length.
__global__ void k_extend_map(const int32_t* __restrict__ known, const int64_t* __restrict__ rank, const uint64_t* __restrict__ hash_of,
                             const int64_t* __restrict__ loc_pool_off, int64_t n_loc, int64_t n_terms,
                             int32_t* __restrict__ map, uint64_t* __restrict__ new_hash, uint32_t* __restrict__ new_term,
                             uint32_t* __restrict__ new_src, uint32_t* __restrict__ new_len) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_loc) return;
    if (known[r] >= 0) { map[r] = known[r]; return; }
    const int64_t s = rank[r];
    map[r] = (int32_t)(n_terms + s);
    new_hash[s] = hash_of[r];
    new_term[s] = (uint32_t)(n_terms + s);
    new_src[s] = (uint32_t)r;
    new_len[s] = (uint32_t)(loc_pool_off[r + 1] - loc_pool_off[r]);
}

__global__ void k_remap(int32_t* __restrict__ ids, int64_t n, const int32_t* __restrict__ map) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ids[i] = map[ids[i]];
}

// New term s: its string goes to the end of the pool, pool_off[n_terms + s + 1] = end of it (off: exclusive scan of
// the new strings' lengths).
__global__ void k_extend_pool(const uint32_t* __restrict__ new_src, const int64_t* __restrict__ off, int64_t n_new,
                              const int64_t* __restrict__ loc_pool_off, const uint8_t* __restrict__ loc_pool,
                              int64_t n_terms, int64_t pool_bytes, int64_t* __restrict__ pool_off, uint8_t* __restrict__ pool) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_new) return;
    const uint32_t r = new_src[s];
    const int64_t a = loc_pool_off[r], n = loc_pool_off[r + 1] - a;
    uint8_t* o = pool + pool_bytes + off[s];
    for (int64_t b = 0; b < n; ++b) o[b] = loc_pool[a + b];
    pool_off[n_terms + s + 1] = pool_bytes + off[s + 1];
}

int report_bad(int bad, const char* who) {
    if (bad & 2) { set_error(std::string(who) + ": byte offsets not non-decreasing"); return BR_ERR_INVALID; }
    if (bad & 4) { set_error(std::string(who) + ": a document of 2 GiB or more"); return BR_ERR_UNSUPPORTED; }
    if (bad & 8) { set_error(std::string(who) + ": two different terms share a 64-bit hash (refusing to merge them)"); return BR_ERR_UNSUPPORTED; }
    return BR_OK;
}

// (start, len) of every token, given the per-document token offsets of tokenize_count
int emit_tokens(StreamScratch& tmp, const uint8_t* text, const int64_t* doc_off, int64_t n_docs, int bigrams,
                const int64_t* doc_tok_off, int64_t n_tok, cudaStream_t st, int64_t** tok_start, uint32_t** tok_len) {
    BR_TRY(tmp.alloc(tok_start, (size_t)n_tok));
    BR_TRY(tmp.alloc(tok_len, (size_t)n_tok));
    if (n_tok > 0) {
        k_tok_emit<<<kNumSMs * 8, 256, 0, st>>>(text, doc_off, doc_tok_off, n_docs, bigrams, *tok_start, *tok_len);
        BR_CUDA(cudaGetLastError());
    }
    return BR_OK;
}

template <class K, class V>
int sort_pairs(StreamScratch& tmp, K** keys, V** vals, int64_t n, int end_bit, cudaStream_t st) {
    if (n <= 1) return BR_OK;
    K* k2 = nullptr;
    V* v2 = nullptr;
    BR_TRY(tmp.alloc(&k2, (size_t)n));
    BR_TRY(tmp.alloc(&v2, (size_t)n));
    cub::DoubleBuffer<K> dk(*keys, k2);
    cub::DoubleBuffer<V> dv(*vals, v2);
    size_t bytes = 0;
    BR_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, n, 0, end_bit, st));
    uint8_t* scratch = nullptr;
    BR_TRY(tmp.alloc(&scratch, bytes + 16));
    BR_CUDA(cub::DeviceRadixSort::SortPairs(scratch, bytes, dk, dv, n, 0, end_bit, st));
    *keys = dk.Current();
    *vals = dv.Current();
    return BR_OK;
}

}  // namespace
}  // namespace br

using namespace br;

extern "C" {

int br_tokenize_count(const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs, int bigrams,
                      int64_t* doc_tok_off_dev, int64_t* n_tokens_host, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    BR_REQUIRE(doc_byte_off_dev && doc_tok_off_dev && n_tokens_host && n_docs >= 0, BR_ERR_INVALID,
               "br_tokenize_count: null pointer / negative n_docs");
    StreamScratch tmp(st);
    uint32_t* counts = nullptr;
    int* d_bad = nullptr;
    BR_TRY(tmp.alloc(&counts, (size_t)n_docs));
    BR_TRY(tmp.alloc(&d_bad, 1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    if (n_docs > 0) {
        k_tok_count<<<kNumSMs * 8, 256, 0, st>>>(text_dev, doc_byte_off_dev, n_docs, bigrams, counts, d_bad);
        BR_CUDA(cudaGetLastError());
    }
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(counts, n_docs, doc_tok_off_dev);
    BR_CUDA(cudaGetLastError());
    int bad = 0;
    BR_CUDA(cudaMemcpyAsync(n_tokens_host, doc_tok_off_dev + n_docs, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_TRY(report_bad(bad, "br_tokenize_count"));
    BR_REQUIRE(*n_tokens_host < (1LL << 31), BR_ERR_UNSUPPORTED, "br_tokenize_count: 2^31 or more tokens in one call");
    return BR_OK;
}

int br_vocab_build(const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs, int bigrams,
                   const int64_t* doc_tok_off_dev, int64_t n_tokens, int32_t* token_ids_dev, void* stream,
                   br_vocab** out) {
    cudaStream_t st = (cudaStream_t)stream;
    BR_REQUIRE(out && doc_byte_off_dev && doc_tok_off_dev && n_docs >= 0, BR_ERR_INVALID, "br_vocab_build: null pointer");
    BR_REQUIRE(n_tokens >= 0 && n_tokens < (1LL << 31), BR_ERR_UNSUPPORTED, "br_vocab_build: 2^31 or more tokens");
    BR_REQUIRE(n_tokens == 0 || token_ids_dev, BR_ERR_INVALID, "br_vocab_build: null token_ids");
    *out = nullptr;
    std::unique_ptr<br_vocab> v(new br_vocab());   // a half-built handle: freed unless released
    BR_CUDA(cudaGetDevice(&v->device));
    StreamScratch tmp(st);
    const int64_t T = n_tokens;

    int64_t* tok_start = nullptr;
    uint32_t *tok_len = nullptr, *idx = nullptr, *block_counts = nullptr;
    uint64_t* hash = nullptr;
    int64_t* block_off = nullptr;
    int* d_bad = nullptr;
    BR_TRY(emit_tokens(tmp, text_dev, doc_byte_off_dev, n_docs, bigrams, doc_tok_off_dev, T, st, &tok_start, &tok_len));
    BR_TRY(tmp.alloc(&hash, (size_t)T));
    BR_TRY(tmp.alloc(&idx, (size_t)T));
    BR_TRY(tmp.alloc(&d_bad, 1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    int64_t V = 0;
    uint32_t *first_tok = nullptr, *run_id = nullptr;
    int32_t* term_of_run = nullptr;
    const int64_t n_blocks = (T + kTile - 1) / kTile;
    if (T > 0) {
        k_tok_hash<<<blocks_for(T, 256), 256, 0, st>>>(text_dev, tok_start, tok_len, T, hash, idx);
        BR_CUDA(cudaGetLastError());
        BR_TRY(sort_pairs(tmp, &hash, &idx, T, 64, st));   // stable: equal hashes keep ascending token index
        BR_TRY(tmp.alloc(&block_counts, (size_t)n_blocks + 1));
        BR_TRY(tmp.alloc(&block_off, (size_t)n_blocks + 2));
        k_head_count<<<(unsigned)n_blocks, kTile, 0, st>>>(hash, T, block_counts);
        BR_CUDA(cudaGetLastError());
        k_exscan<uint32_t><<<1, 1024, 0, st>>>(block_counts, n_blocks, block_off);
        BR_CUDA(cudaGetLastError());
        BR_CUDA(cudaMemcpyAsync(&V, block_off + n_blocks, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaStreamSynchronize(st));
    }
    v->n_terms = V;
    BR_TRY(v->hash_sorted.alloc((size_t)V));
    BR_TRY(v->term_sorted.alloc((size_t)V));
    BR_TRY(v->pool_off.alloc((size_t)V + 1));
    if (V > 0) {
        BR_TRY(tmp.alloc(&first_tok, (size_t)V));
        BR_TRY(tmp.alloc(&run_id, (size_t)V));
        k_head_emit<<<(unsigned)n_blocks, kTile, 0, st>>>(hash, idx, T, block_off, v->hash_sorted, first_tok, run_id);
        BR_CUDA(cudaGetLastError());
        // term id = rank of the run's first occurrence (dict insertion order of the reference's build loop)
        uint32_t* first_unsorted = nullptr;
        BR_TRY(tmp.alloc(&first_unsorted, (size_t)V));
        BR_CUDA(cudaMemcpyAsync(first_unsorted, first_tok, sizeof(uint32_t) * (size_t)V, cudaMemcpyDeviceToDevice, st));
        uint32_t* first_by_rank = first_tok;   // sorted in place (double buffer) below
        int bits = 1;
        while ((1LL << bits) < T) ++bits;
        BR_TRY(sort_pairs(tmp, &first_by_rank, &run_id, V, bits, st));
        term_of_run = v->term_sorted;
        k_rank_scatter<<<blocks_for(V, 256), 256, 0, st>>>(run_id, V, term_of_run);
        BR_CUDA(cudaGetLastError());
        k_assign<<<(unsigned)n_blocks, kTile, 0, st>>>(text_dev, tok_start, tok_len, hash, idx, T, block_off,
                                                       first_unsorted, term_of_run, token_ids_dev, d_bad);
        BR_CUDA(cudaGetLastError());
        // vocabulary strings
        uint32_t* clen = nullptr;
        BR_TRY(tmp.alloc(&clen, (size_t)V));
        k_pool_len<<<blocks_for(V, 256), 256, 0, st>>>(text_dev, tok_start, tok_len, first_by_rank, V, clen);
        BR_CUDA(cudaGetLastError());
        k_exscan<uint32_t><<<1, 1024, 0, st>>>(clen, V, v->pool_off);
        BR_CUDA(cudaGetLastError());
        int bad = 0;
        BR_CUDA(cudaMemcpyAsync(&v->pool_bytes, v->pool_off + V, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaStreamSynchronize(st));
        BR_TRY(report_bad(bad, "br_vocab_build"));
        BR_TRY(v->pool.alloc((size_t)v->pool_bytes));
        k_pool_fill<<<blocks_for(V, 256), 256, 0, st>>>(text_dev, tok_start, tok_len, first_by_rank, V, v->pool_off, v->pool);
        BR_CUDA(cudaGetLastError());
    } else {
        BR_CUDA(cudaMemsetAsync(v->pool_off, 0, sizeof(int64_t), st));
        BR_TRY(v->pool.alloc(0));
    }
    BR_CUDA(cudaStreamSynchronize(st));   // temporaries are freed when tmp goes out of scope
    *out = v.release();
    return BR_OK;
}

int br_vocab_lookup(const br_vocab* v, const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs,
                    int bigrams, const int64_t* doc_tok_off_dev, int64_t n_tokens, int32_t* token_ids_dev, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    BR_REQUIRE(v && doc_byte_off_dev && doc_tok_off_dev, BR_ERR_INVALID, "br_vocab_lookup: null pointer");
    BR_REQUIRE(n_tokens >= 0 && n_tokens < (1LL << 31), BR_ERR_UNSUPPORTED, "br_vocab_lookup: 2^31 or more tokens");
    if (n_tokens == 0) return BR_OK;
    BR_REQUIRE(token_ids_dev, BR_ERR_INVALID, "br_vocab_lookup: null token_ids");
    StreamScratch tmp(st);
    int64_t* tok_start = nullptr;
    uint32_t* tok_len = nullptr;
    BR_TRY(emit_tokens(tmp, text_dev, doc_byte_off_dev, n_docs, bigrams, doc_tok_off_dev, n_tokens, st, &tok_start, &tok_len));
    k_lookup<<<blocks_for(n_tokens, 256), 256, 0, st>>>(text_dev, tok_start, tok_len, n_tokens, v->hash_sorted,
                                                        v->term_sorted, v->n_terms, v->pool_off, v->pool, token_ids_dev);
    BR_CUDA(cudaGetLastError());
    BR_CUDA(cudaStreamSynchronize(st));
    return BR_OK;
}

// The new text gets a vocabulary of its own (br_vocab_build: its terms in first-occurrence order, its tokens' local ids);
// its terms are looked up in v, the ones not found are numbered after v's terms in local order, the tokens are
// remapped, the new strings appended to the pool and the new (hash, id) pairs sorted into the hash table.  The grown
// tables are complete before they replace v's.
int br_vocab_extend(br_vocab* v, const uint8_t* text_dev, const int64_t* doc_byte_off_dev, int64_t n_docs, int bigrams,
                    const int64_t* doc_tok_off_dev, int64_t n_tokens, int32_t* token_ids_dev, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    BR_REQUIRE(v && doc_byte_off_dev && doc_tok_off_dev && n_docs >= 0, BR_ERR_INVALID, "br_vocab_extend: null pointer");
    BR_REQUIRE(n_tokens >= 0 && n_tokens < (1LL << 31), BR_ERR_UNSUPPORTED, "br_vocab_extend: 2^31 or more tokens");
    BR_REQUIRE(n_tokens == 0 || token_ids_dev, BR_ERR_INVALID, "br_vocab_extend: null token_ids");
    if (n_tokens == 0) return BR_OK;
    BR_CUDA(cudaSetDevice(v->device));
    br_vocab* loc_raw = nullptr;
    BR_TRY(br_vocab_build(text_dev, doc_byte_off_dev, n_docs, bigrams, doc_tok_off_dev, n_tokens, token_ids_dev, stream,
                          &loc_raw));
    std::unique_ptr<br_vocab> loc(loc_raw);
    const int64_t L = loc->n_terms, V = v->n_terms;
    StreamScratch tmp(st);
    int32_t *known = nullptr, *map = nullptr;
    uint32_t* is_new = nullptr;
    uint64_t* hash_of = nullptr;
    int64_t* rank = nullptr;
    int* d_bad = nullptr;
    BR_TRY(tmp.alloc(&known, (size_t)L));
    BR_TRY(tmp.alloc(&map, (size_t)L));
    BR_TRY(tmp.alloc(&is_new, (size_t)L));
    BR_TRY(tmp.alloc(&hash_of, (size_t)L));
    BR_TRY(tmp.alloc(&rank, (size_t)L + 1));
    BR_TRY(tmp.alloc(&d_bad, 1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    k_extend_find<<<blocks_for(L, 256), 256, 0, st>>>(loc->hash_sorted, loc->term_sorted, L, loc->pool_off, loc->pool,
                                                      v->hash_sorted, v->term_sorted, V, v->pool_off, v->pool, known,
                                                      is_new, hash_of, d_bad);
    BR_CUDA(cudaGetLastError());
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(is_new, L, rank);
    BR_CUDA(cudaGetLastError());
    int64_t n_new = 0;
    int bad = 0;
    BR_CUDA(cudaMemcpyAsync(&n_new, rank + L, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_TRY(report_bad(bad, "br_vocab_extend"));
    BR_REQUIRE(V + n_new < (1LL << 31), BR_ERR_UNSUPPORTED, "br_vocab_extend: 2^31 or more terms");

    const int64_t W = V + n_new;
    uint64_t* cat_hash = nullptr;
    uint32_t *cat_term = nullptr, *new_src = nullptr, *new_len = nullptr;
    int64_t* new_off = nullptr;
    BR_TRY(tmp.alloc(&cat_hash, (size_t)W));
    BR_TRY(tmp.alloc(&cat_term, (size_t)W));
    BR_TRY(tmp.alloc(&new_src, (size_t)n_new));
    BR_TRY(tmp.alloc(&new_len, (size_t)n_new));
    BR_TRY(tmp.alloc(&new_off, (size_t)n_new + 1));
    if (V > 0) {
        BR_CUDA(cudaMemcpyAsync(cat_hash, v->hash_sorted, sizeof(uint64_t) * (size_t)V, cudaMemcpyDeviceToDevice, st));
        BR_CUDA(cudaMemcpyAsync(cat_term, v->term_sorted, sizeof(int32_t) * (size_t)V, cudaMemcpyDeviceToDevice, st));
    }
    k_extend_map<<<blocks_for(L, 256), 256, 0, st>>>(known, rank, hash_of, loc->pool_off, L, V, map, cat_hash + V,
                                                     cat_term + V, new_src, new_len);
    BR_CUDA(cudaGetLastError());
    k_remap<<<blocks_for(n_tokens, 256), 256, 0, st>>>(token_ids_dev, n_tokens, map);
    BR_CUDA(cudaGetLastError());
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(new_len, n_new, new_off);
    BR_CUDA(cudaGetLastError());
    int64_t new_bytes = 0;
    BR_CUDA(cudaMemcpyAsync(&new_bytes, new_off + n_new, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    // the hash tables' entries are distinct (a new term's hash is not in v), so sorting the concatenation by hash gives
    // exactly the table br_vocab_build makes over old text + new text
    BR_TRY(sort_pairs(tmp, &cat_hash, &cat_term, W, 64, st));
    BR_CUDA(cudaStreamSynchronize(st));

    DevArray<uint64_t> hash_sorted;
    DevArray<int32_t> term_sorted;
    DevArray<int64_t> pool_off;
    DevArray<uint8_t> pool;
    BR_TRY(hash_sorted.alloc((size_t)W));
    BR_TRY(term_sorted.alloc((size_t)W));
    BR_TRY(pool_off.alloc((size_t)W + 1));
    BR_TRY(pool.alloc((size_t)(v->pool_bytes + new_bytes)));
    BR_CUDA(cudaMemcpyAsync(hash_sorted, cat_hash, sizeof(uint64_t) * (size_t)W, cudaMemcpyDeviceToDevice, st));
    k_u32_to_i32<<<blocks_for(W, 256), 256, 0, st>>>(cat_term, W, term_sorted);
    BR_CUDA(cudaGetLastError());
    BR_CUDA(cudaMemcpyAsync(pool_off, v->pool_off, sizeof(int64_t) * (size_t)(V + 1), cudaMemcpyDeviceToDevice, st));
    if (v->pool_bytes > 0)
        BR_CUDA(cudaMemcpyAsync(pool, v->pool, (size_t)v->pool_bytes, cudaMemcpyDeviceToDevice, st));
    if (n_new > 0) {
        k_extend_pool<<<blocks_for(n_new, 256), 256, 0, st>>>(new_src, new_off, n_new, loc->pool_off, loc->pool, V,
                                                              v->pool_bytes, pool_off, pool);
        BR_CUDA(cudaGetLastError());
    }
    BR_CUDA(cudaStreamSynchronize(st));

    // nothing below can fail
    v->hash_sorted = std::move(hash_sorted);
    v->term_sorted = std::move(term_sorted);
    v->pool_off = std::move(pool_off);
    v->pool = std::move(pool);
    v->n_terms = W;
    v->pool_bytes += new_bytes;
    return BR_OK;
}

int br_vocab_stats(const br_vocab* v, int64_t* n_terms, int64_t* pool_bytes) {
    BR_REQUIRE(v, BR_ERR_INVALID, "br_vocab_stats: null handle");
    if (n_terms) *n_terms = v->n_terms;
    if (pool_bytes) *pool_bytes = v->pool_bytes;
    return BR_OK;
}

int br_vocab_export(const br_vocab* v, int64_t* pool_off_host, uint8_t* pool_host) {
    BR_REQUIRE(v && pool_off_host, BR_ERR_INVALID, "br_vocab_export: null pointer");
    BR_CUDA(cudaMemcpy(pool_off_host, v->pool_off, sizeof(int64_t) * (size_t)(v->n_terms + 1), cudaMemcpyDeviceToHost));
    if (v->pool_bytes > 0) {
        BR_REQUIRE(pool_host, BR_ERR_INVALID, "br_vocab_export: null pool");
        BR_CUDA(cudaMemcpy(pool_host, v->pool, (size_t)v->pool_bytes, cudaMemcpyDeviceToHost));
    }
    return BR_OK;
}

int br_vocab_import(const int64_t* pool_off_host, const uint8_t* pool_host, int64_t n_terms, void* stream, br_vocab** out) {
    cudaStream_t st = (cudaStream_t)stream;
    BR_REQUIRE(out && pool_off_host && n_terms >= 0 && n_terms < (1LL << 31), BR_ERR_INVALID, "br_vocab_import: bad arguments");
    *out = nullptr;
    std::unique_ptr<br_vocab> v(new br_vocab());   // a half-built handle: freed unless released
    BR_CUDA(cudaGetDevice(&v->device));
    const int64_t V = n_terms;
    v->n_terms = V;
    v->pool_bytes = pool_off_host[V];
    BR_REQUIRE(pool_off_host[0] == 0 && v->pool_bytes >= 0, BR_ERR_INVALID, "br_vocab_import: bad pool offsets");
    BR_TRY(v->hash_sorted.alloc((size_t)V));
    BR_TRY(v->term_sorted.alloc((size_t)V));
    BR_TRY(v->pool_off.alloc((size_t)V + 1));
    BR_TRY(v->pool.alloc((size_t)v->pool_bytes));
    BR_CUDA(cudaMemcpyAsync(v->pool_off, pool_off_host, sizeof(int64_t) * (size_t)(V + 1), cudaMemcpyHostToDevice, st));
    if (v->pool_bytes > 0)
        BR_CUDA(cudaMemcpyAsync(v->pool, pool_host, (size_t)v->pool_bytes, cudaMemcpyHostToDevice, st));
    StreamScratch tmp(st);
    if (V > 0) {
        uint64_t* hash = nullptr;
        uint32_t* term = nullptr;
        int* d_bad = nullptr;
        BR_TRY(tmp.alloc(&hash, (size_t)V));
        BR_TRY(tmp.alloc(&term, (size_t)V));
        BR_TRY(tmp.alloc(&d_bad, 1));
        BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
        k_pool_hash<<<blocks_for(V, 256), 256, 0, st>>>(v->pool, v->pool_off, V, hash, term);
        BR_CUDA(cudaGetLastError());
        BR_TRY(sort_pairs(tmp, &hash, &term, V, 64, st));
        k_dup_check<<<blocks_for(V, 256), 256, 0, st>>>(hash, V, d_bad);
        BR_CUDA(cudaGetLastError());
        BR_CUDA(cudaMemcpyAsync(v->hash_sorted, hash, sizeof(uint64_t) * (size_t)V, cudaMemcpyDeviceToDevice, st));
        k_u32_to_i32<<<blocks_for(V, 256), 256, 0, st>>>(term, V, v->term_sorted);
        BR_CUDA(cudaGetLastError());
        int bad = 0;
        BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaStreamSynchronize(st));
        BR_REQUIRE(!(bad & 8), BR_ERR_INVALID, "br_vocab_import: duplicate term (or 64-bit hash collision) in the vocabulary");
    }
    BR_CUDA(cudaStreamSynchronize(st));
    *out = v.release();
    return BR_OK;
}

void br_vocab_destroy(br_vocab* v) { delete v; }

}  // extern "C"
