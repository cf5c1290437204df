// br_query.cu - query-time kernels of the dense ("generic") BM25 path and the shared tail:
//
//   k_prep_queries   per query: drop OOV terms, de-duplicate (set(query), bm25_ranking.ipynb:193)
//                    or keep multiplicities (team_run1.py:183), sort by term id, prefix df
//   k_score_dense    term-at-a-time scatter-add of packed postings into fp32 [nq, N] accumulators
//                    (get_scores, bm25_ranking.ipynb:191-204)
//   k_select_radix   per query row: exact k-th largest fp32 score by 3-pass radix select, then the
//                    candidate band  s >= kth - 1e-5*|kth|   (retrieve_top_n, :206-213)
//   k_emit_cands     band members -> candidate list (doc-id order; zero-score tail in doc-id order)
//   k_rescore<F>     exact float64 re-evaluation of formula F (BM25, TF-IDF cosine, V3 re-rank) for every candidate,
//                    candidates in per-query ranges cand_off (dense path, br_rescore_docs, br_rerank_v3_scores)
//   k_rescore_heads<F>  the same over fixed-stride per-query regions with a live count, one CTA per query (tiled
//                    path, br_fuse_linear)
//   k_final_select   (score64 desc, doc id asc) order, top-k, duplicate ids removed
// k_select_radix, k_emit_cands and the tiled path's k_seed_thr take a doc filter; a null row table means unfiltered.
//
// Why a band + float64 re-score: the reference ranks float64 scores; fp32 accumulation can swap
// near-ties.  Every doc outside the band has fp32 score < kth32*(1-1e-5), hence (fp32 error of a
// <=64-term positive sum is < 4e-6 relative) a float64 score below that of the k band members that
// define kth32 - so the true top-k is inside the band, and re-scoring the band in float64 gives the
// reference's ranking exactly (DESIGN.md, "exactness").  A query with a term of negative idf (okapi_no_plus1) sums
// weights of both signs: its band also reaches kth32 - slack, an absolute bound of the fp32 error, and a hit row tells
// its docs with a hit from those without (k_select_radix).
#include <math_constants.h>

#include <utility>

#include "br_common.cuh"
#include "br_kernels.cuh"
#include "br_query.cuh"

namespace br {

// ------------------------------------------------------------------------------------------
// query preparation
// ------------------------------------------------------------------------------------------
constexpr int SCORE_CHUNK = 8192;

__global__ void k_prep_queries(const int32_t* __restrict__ q_terms, const int32_t* __restrict__ q_off, int32_t nq,
                               int32_t vocab, const int64_t* __restrict__ row_ptr, const int8_t* __restrict__ sig_bit, int dedup,
                               const double* __restrict__ idf, const float* __restrict__ amax, PrepView v) {
    const int lane = threadIdx.x & 31;
    const int q = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (q >= nq) return;
    const int32_t off = q_off[q];
    int32_t M = q_off[q + 1] - off;
    if (off < 0 || M < 0 || off + M > v.t_cap) {         // offsets beyond the caller's n_terms: treated as an empty query
        if (lane == 0) atomicOr(v.bad, 1);
        M = 0;
    }
    // phase 1: validity, ordered compaction into o_terms
    int32_t n_valid = 0;
    for (int32_t base = 0; base < M; base += 32) {
        const int32_t i = base + lane;
        int32_t t = -1;
        bool ok = false;
        if (i < M) {
            t = q_terms[off + i];
            ok = t >= 0 && t < vocab && row_ptr[t + 1] > row_ptr[t];
        }
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (ok) v.o_terms[off + n_valid + __popc(m & ((1u << lane) - 1))] = t;
        n_valid += __popc(m);
    }
    __syncwarp();
    // phase 2: first-occurrence flag + multiplicity among the valid terms
    for (int32_t i = lane; i < n_valid; i += 32) {
        const int32_t t = v.o_terms[off + i];
        int32_t mult = 0;
        bool first = true;
        for (int32_t j = 0; j < n_valid; ++j) {
            const bool eq = v.o_terms[off + j] == t;
            mult += eq ? 1 : 0;
            if (eq && j < i) first = false;
        }
        v.tmp[off + i] = first ? mult : 0;
    }
    __syncwarp();
    // phase 3: rank among the distinct terms -> ascending unique list
    int32_t n_uniq = 0;
    uint32_t sig = 0;
    for (int32_t base = 0; base < n_valid; base += 32) {
        const int32_t i = base + lane;
        const bool first = i < n_valid && v.tmp[off + i] > 0;
        if (first) {
            const int32_t t = v.o_terms[off + i];
            const int sb = sig_bit ? sig_bit[t] : -1;
            if (sb >= 0) sig |= 1u << (31 - sb);
            int32_t rank = 0;
            for (int32_t j = 0; j < n_valid; ++j) rank += (v.tmp[off + j] > 0 && v.o_terms[off + j] < t) ? 1 : 0;
            v.u_terms[off + rank] = t;
            v.u_mult[off + rank] = dedup ? 1 : v.tmp[off + i];
        }
        n_uniq += __popc(__ballot_sync(0xffffffffu, first));
    }
    __syncwarp();
    for (int o = 16; o > 0; o >>= 1) sig |= __shfl_xor_sync(0xffffffffu, sig, o);
    if (lane == 0) {
        v.sig[q] = sig;
        int64_t cum = 0;
        float wsum = 0.f;
        bool neg = false;
        for (int32_t i = 0; i < n_uniq; ++i) {
            const int32_t t = v.u_terms[off + i];
            v.u_cum[off + i] = cum;
            cum += row_ptr[t + 1] - row_ptr[t];
            if (amax) {
                neg |= idf[t] < 0.0;
                wsum += (float)v.u_mult[off + i] * amax[t];
            }
        }
        v.slack[q] = neg ? ldexpf((float)(2 * n_uniq + 6), -24) * wsum : 0.f;
        v.u_cnt[q] = n_uniq;
        v.o_cnt[q] = n_valid;
        v.P[q] = cum;
        v.n_chunks[q] = (uint32_t)((cum + SCORE_CHUNK - 1) / SCORE_CHUNK);
    }
}

// Hit rows of the dense path's queries with a term of negative idf (PrepView::slack[q] > 0): bit (d & 31) of word
// (d >> 5) of the query's row is set when doc d holds at least one of its terms.  With mixed signs a doc's fp32 sum can
// be exactly 0 while its float64 score is not, so "fp32 score 0" no longer means "no hit" for such a query.  slack ==
// nullptr (other variants, the TF-IDF weight table): no query has a row.  Rows follow the pass's query order.
struct HitRows {
    const float* slack;
    uint32_t* bits;
    int64_t words;
    __device__ __forceinline__ uint32_t* row_of(int q, int row) const {
        return slack && slack[q] > 0.f ? bits + (int64_t)row * words : nullptr;
    }
};
// hr: the query's hit row (nullptr: a query whose weights are all >= 0, where fp32 score 0 means no hit)
__device__ __forceinline__ bool no_hit(const uint32_t* hr, float s, uint32_t doc) {
    return hr ? ((hr[doc >> 5] >> (doc & 31)) & 1u) == 0u : s == 0.0f;
}

// ------------------------------------------------------------------------------------------
// dense scoring: one work item = SCORE_CHUNK consecutive postings of one query's concatenated lists
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_score_dense(const br_posting* __restrict__ post,
                                                     const int64_t* __restrict__ row_ptr,
                                                     const int32_t* __restrict__ q_off, PrepView v,
                                                     const int64_t* __restrict__ chunk_start, int32_t q_begin,
                                                     int32_t nq, float* __restrict__ out, int64_t n_docs, HitRows h) {
    const int64_t w_begin = chunk_start[q_begin], w_end = chunk_start[q_begin + nq];
    for (int64_t w = w_begin + blockIdx.x; w < w_end; w += gridDim.x) {
        // query of this work item: last q with chunk_start[q] <= w
        int32_t lo = q_begin, hi = q_begin + nq;
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (chunk_start[mid] <= w) lo = mid; else hi = mid;
        }
        const int32_t q = lo;
        const int32_t off = q_off[q], nt = v.u_cnt[q];
        const int64_t e0 = (w - chunk_start[q]) * SCORE_CHUNK;
        const int64_t e1 = min(e0 + (int64_t)SCORE_CHUNK, v.P[q]);
        float* row = out + (int64_t)(q - q_begin) * n_docs;
        uint32_t* hr = h.row_of(q, q - q_begin);
        for (int64_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
            int32_t a = 0, b = nt;  // last term index with u_cum <= e
            while (b - a > 1) {
                const int32_t mid = (a + b) >> 1;
                if (v.u_cum[off + mid] <= e) a = mid; else b = mid;
            }
            const int32_t t = v.u_terms[off + a];
            const br_posting p = post[row_ptr[t] + (e - v.u_cum[off + a])];
            atomicAdd(row + p.doc, p.w * (float)v.u_mult[off + a]);
            if (hr) atomicOr(hr + (p.doc >> 5), 1u << (p.doc & 31));
        }
    }
}

// ------------------------------------------------------------------------------------------
// radix select
// ------------------------------------------------------------------------------------------
// nh: the doc has no hit (no_hit); under positive_only such a doc gets key 0, below every doc with a hit
__device__ __forceinline__ uint32_t score_key(float s, bool nh, int positive_only) {
    if (positive_only && nh) return 0u;
    const uint32_t u = __float_as_uint(s);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_score(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct SelView {
    float* lo;         // [nq] band lower bound
    int32_t* mode;     // [nq] 0 band, 1 band over docs with a hit + zero fill, 2 all (with a hit, positive_only)
    int32_t* zfill;    // [nq] number of docs without a hit to take in doc-id order (mode 1)
    int64_t* cnt;      // [nq] number of candidates the emit kernel writes
};

constexpr int SEL_T = 1024;

// A doc the query's filter row excludes gets key 0, below every allowed doc, so kth_key == 0 means "fewer than k
// allowed docs (with a hit, for positive_only)": mode 2 then takes every allowed doc (with a hit).  Disallowed docs are
// neither counted nor emitted, so the zero-score tail of mode 1 is made of allowed docs in doc-id order.  Unfiltered,
// kth_key == 0 needs positive_only: without it no non-NaN score has key 0, and k_rem <= n_docs makes the k-th key a
// doc's own key.  Two CTAs per SM (at most 32 registers): the filter test must not halve the occupancy of the unfiltered
// select.
// A query with a term of negative idf (slack sl > 0, hit row hr) widens the band to kth - sl, which bounds the fp32
// error of a mixed-sign sum where the relative band does not.  Once the band reaches 0 (mode 1) it takes every doc WITH
// a hit whose fp32 score is >= lo, fp32 zeros included, and fills with docs WITHOUT a hit in doc-id order: all of them
// score exactly 0, and at most k minus the docs with fp32 score > sl (surely > 0 in float64) belong to the top k.  Under
// positive_only a doc with a hit can score exactly 0 in float64 (dropped later, by k_final_select); only docs with
// |fp32| <= sl can, so the select looks for the (k + their number)-th key instead of the k-th.  For every other query
// (sl == 0, fp32 zero == no hit) each rule reduces to the positive-weight one.
__global__ void __launch_bounds__(SEL_T, 2) k_select_radix(const float* __restrict__ scores, int64_t n_docs, int32_t k,
                                                        int positive_only, SelView sv, int32_t q_begin,
                                                        const int32_t* __restrict__ n_terms, DocFilter f, HitRows h) {
    __shared__ uint32_t hist[2048];
    __shared__ uint32_t s_bin, s_above;
    __shared__ unsigned long long s_cnt[3];
    const float* row = scores + (int64_t)blockIdx.x * n_docs;
    const int q = q_begin + blockIdx.x;
    const uint32_t* fr = f.row ? f.row_of(q) : nullptr;
    const uint32_t* hr = h.row_of(q, blockIdx.x);
    const float sl = hr ? h.slack[q] : 0.f;
    uint32_t prefix = 0, mask = 0;
    int64_t k_sel = k;
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    if (hr && positive_only) {
        uint32_t n_amb = 0;
        for (int64_t i = threadIdx.x; i < n_docs; i += SEL_T)
            n_amb += doc_allowed(fr, (uint32_t)i) && !no_hit(hr, row[i], (uint32_t)i) && fabsf(row[i]) <= sl;
        n_amb = __reduce_add_sync(0xffffffffu, n_amb);
        if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt[2], (unsigned long long)n_amb);
        __syncthreads();
        k_sel += (int64_t)s_cnt[2];
    }
    uint32_t k_rem = (uint32_t)min(k_sel, n_docs);
#pragma unroll 1
    for (int pass = 0; pass < 3; ++pass) {
        const int shift = pass == 0 ? 21 : pass == 1 ? 10 : 0, nb = pass == 2 ? 1024 : 2048;
        for (int i = threadIdx.x; i < 2048; i += SEL_T) hist[i] = 0;
        __syncthreads();
        for (int64_t i = threadIdx.x; i < n_docs; i += SEL_T) {
            const float s = row[i];
            const uint32_t u = doc_allowed(fr, (uint32_t)i) ? score_key(s, no_hit(hr, s, (uint32_t)i), positive_only) : 0u;
            if ((u & mask) == prefix) atomicAdd(&hist[(u >> shift) & (nb - 1)], 1u);
        }
        __syncthreads();
        // bins from the top: thread t owns reversed bins 2t, 2t+1
        const int r0 = 2 * threadIdx.x, r1 = r0 + 1;
        const uint32_t v0 = r0 < nb ? hist[nb - 1 - r0] : 0u, v1 = r1 < nb ? hist[nb - 1 - r1] : 0u;
        uint32_t total;
        const uint32_t ex = block_excl_scan(v0 + v1, &total);
        if (ex < k_rem && k_rem <= ex + v0) { s_bin = nb - 1 - r0; s_above = ex; }
        else if (ex + v0 < k_rem && k_rem <= ex + v0 + v1) { s_bin = nb - 1 - r1; s_above = ex + v0; }
        __syncthreads();
        prefix |= s_bin << shift;
        mask |= (uint32_t)(nb - 1) << shift;
        k_rem -= s_above;
        __syncthreads();
    }
    // prefix = key of the k-th largest score
    const uint32_t kth_key = prefix;
    int mode = 0;
    float lo = 0.f;
    if (kth_key == 0u) {
        mode = 2;                                   // fewer than k allowed docs with a hit: take them all
    } else {
        const float kth = key_score(kth_key);
        // fp32 error of an n-term sum grows with n: widen the band for unusually long queries
        const float band = kBandRel * (float)max(1, (n_terms[q] + 31) / 32);
        lo = fminf(kth - band * fabsf(kth), kth - sl);
        if (!positive_only && lo <= 0.0f) mode = 1; // the band reaches the zero-score docs: zero tail in doc order
    }
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    unsigned long long c_band = 0, c_sure = 0, c_zero = 0;
    for (int64_t i = threadIdx.x; i < n_docs; i += SEL_T) {
        const float s = row[i];
        const bool ok = doc_allowed(fr, (uint32_t)i);
        const bool nh = no_hit(hr, s, (uint32_t)i);
        if (mode == 2) c_band += (ok && (!positive_only || !nh));
        else if (mode == 1) { c_band += (ok && s >= lo && !nh); c_sure += (ok && s > sl); c_zero += (ok && nh); }
        else c_band += (ok && s >= lo && !(positive_only && nh));
    }
    for (int o = 16; o > 0; o >>= 1) {
        c_band += __shfl_xor_sync(0xffffffffu, c_band, o);
        c_sure += __shfl_xor_sync(0xffffffffu, c_sure, o);
        c_zero += __shfl_xor_sync(0xffffffffu, c_zero, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_cnt[0], c_band); atomicAdd(&s_cnt[1], c_sure); atomicAdd(&s_cnt[2], c_zero); }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int64_t kk = min((int64_t)k, n_docs);
        sv.lo[q] = lo;
        sv.mode[q] = mode;
        const int64_t zfill = mode == 1 ? min(kk - (int64_t)s_cnt[1], (int64_t)s_cnt[2]) : 0;
        sv.zfill[q] = (int32_t)zfill;
        sv.cnt[q] = (int64_t)s_cnt[0] + zfill;
    }
}

__global__ void __launch_bounds__(SEL_T) k_emit_cands(const float* __restrict__ scores, int64_t n_docs,
                                                      int positive_only, SelView sv, int32_t q_begin,
                                                      const int64_t* __restrict__ cand_off, int32_t* __restrict__ cand,
                                                      DocFilter f, HitRows h) {
    const float* row = scores + (int64_t)blockIdx.x * n_docs;
    const int q = q_begin + blockIdx.x;
    const uint32_t* fr = f.row ? f.row_of(q) : nullptr;
    const uint32_t* hr = h.row_of(q, blockIdx.x);
    const int mode = sv.mode[q];
    const float lo = sv.lo[q];
    const uint32_t zfill = (uint32_t)sv.zfill[q];
    int32_t* out = cand + cand_off[q];
    uint32_t n_out = 0, n_zero = 0;   // running totals (identical in all threads)
    for (int64_t base = 0; base < n_docs; base += SEL_T) {
        const int64_t i = base + threadIdx.x;
        const float s = i < n_docs ? row[i] : -CUDART_INF_F;
        bool take, zero = false;
        const bool ok = i < n_docs && doc_allowed(fr, (uint32_t)i);
        const bool nh = ok && no_hit(hr, s, (uint32_t)i);
        if (mode == 2) take = ok && (!positive_only || !nh);
        else if (mode == 1) { take = ok && s >= lo && !nh; zero = nh; }
        else take = ok && s >= lo && !(positive_only && nh);
        uint32_t total, ztotal = 0, zex = 0;
        if (mode == 1) {
            zex = block_excl_scan(zero ? 1u : 0u, &ztotal);
            if (zero && n_zero + zex < zfill) take = true;
        }
        const uint32_t ex = block_excl_scan(take ? 1u : 0u, &total);
        if (take) out[n_out + ex] = (int32_t)i;
        n_out += total;
        n_zero += ztotal;
    }
}

// ------------------------------------------------------------------------------------------
// exact float64 re-score of candidates
// ------------------------------------------------------------------------------------------
struct RescoreIndex {
    const br_posting* post;
    const uint16_t* tf;
    const int64_t* row_ptr;
    const uint32_t* dl;
    const double* idf;
    const double* inv_norm;   // 1/||d|| of the TF-IDF doc vectors (Formula::COS only)
    const int32_t* hot_slot;
    const uint32_t* skip;
    int32_t n_sub;
    int sub_shift;
    double avgdl, k1, b;
    int variant;
};

// Index of posting (t, doc) in the packed lists, -1 when doc does not contain t.  Hot terms use the skip table to narrow
// the search to one sub-range.
__device__ __forceinline__ int64_t find_posting(const RescoreIndex& r, int32_t t, uint32_t doc) {
    const int64_t base = r.row_ptr[t];
    int64_t lo = base, hi = r.row_ptr[t + 1];
    const int32_t slot = r.skip ? r.hot_slot[t] : -1;
    if (slot >= 0) {
        const uint32_t* sk = r.skip + (int64_t)slot * (r.n_sub + 1) + (doc >> r.sub_shift);
        lo = base + sk[0];
        hi = base + sk[1];
    }
    const int64_t stop = hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (r.post[mid].doc < doc) lo = mid + 1; else hi = mid;
    }
    return lo < stop && r.post[lo].doc == doc ? lo : -1;
}

// BM25: the reference loop body (bm25_ranking.ipynb:199-203) doc-at-a-time; terms are visited in the given order
// (ascending id / query order) so the sum is reproducible.
__device__ __forceinline__ double score_bm25(const RescoreIndex& r, const int32_t* __restrict__ terms, int32_t nt,
                                             uint32_t doc) {
    double s = 0.0;
    const double dld = (double)r.dl[doc];
    for (int32_t i = 0; i < nt; ++i) {
        const int32_t t = terms[i];
        const int64_t p = find_posting(r, t, doc);
        if (p >= 0) s = __dadd_rn(s, bm25_contrib(r.idf[t], (double)r.tf[p], dld, r.avgdl, r.k1, r.b, r.variant));
    }
    return s;
}

// TF-IDF cosine with the reference's mixed precision (cosine_similarity_bm25_reranking.py:88,121-126,210-226): doc
// entries float32(tf*idf) scaled by the float64 1/doc_norm, query entries float32(float32(idf) * float32(1/||q||)),
// products and sum in float64, terms in ascending id.  ||q|| is a float32 BLAS dot in the reference (platform-dependent
// last bit); here float32(sqrt(float64 sum)).
__device__ __forceinline__ double score_cos(const RescoreIndex& r, const int32_t* __restrict__ terms, int32_t nt,
                                            uint32_t doc) {
    double n2 = 0.0;
    for (int32_t i = 0; i < nt; ++i) { const double x = (double)(float)r.idf[terms[i]]; n2 += x * x; }
    const float inv_q = 1.0f / (float)sqrt(n2);
    const double inv_d = r.inv_norm[doc];
    double s = 0.0;
    for (int32_t i = 0; i < nt; ++i) {
        const int32_t t = terms[i];
        const int64_t p = find_posting(r, t, doc);
        if (p < 0 || r.tf[p] == 0) continue;
        const double e = (double)(float)((double)r.tf[p] * r.idf[t]);
        const double qn = (double)((float)r.idf[t] * inv_q);
        s = __dadd_rn(s, __dmul_rn(__dmul_rn(e, inv_d), qn));
    }
    return s;
}

// "V3" re-rank: bm25_score, cosine_similarity_bm25_reranking.py:185-195
//   doc_length = sum of the tf of the query's term occurrences in this doc (:187)
//   score += idf * ((tf*(k1+1)) / (tf + k1*(1 - b + b*(doc_length/avgdl))))   for every occurrence whose
//   term is in the corpus (duplicates counted, idf without +1)
__device__ __forceinline__ double score_v3(const RescoreIndex& r, const int32_t* __restrict__ terms, int32_t nt,
                                           uint32_t doc) {
    int64_t doc_length = 0;
    for (int32_t i = 0; i < nt; ++i) {
        const int64_t p = find_posting(r, terms[i], doc);
        doc_length += p >= 0 ? r.tf[p] : 0;
    }
    const double norm = __dadd_rn(__dsub_rn(1.0, r.b), __dmul_rn(r.b, __ddiv_rn((double)doc_length, r.avgdl)));
    const double kn = __dmul_rn(r.k1, norm);
    double s = 0.0;
    for (int32_t i = 0; i < nt; ++i) {
        const int32_t t = terms[i];
        const int64_t p = find_posting(r, t, doc);
        const double tf = p >= 0 ? (double)r.tf[p] : 0.0;
        const double num = __dmul_rn(tf, __dadd_rn(r.k1, 1.0));
        const double den = __dadd_rn(tf, kn);
        s = __dadd_rn(s, __dmul_rn(r.idf[t], __ddiv_rn(num, den)));
    }
    return s;
}

// The terms formula F sums over for query q: BM25 the distinct terms ascending (dedup) or the occurrences in query
// order; COS the distinct terms; V3 the occurrences.
template <Formula F>
__device__ __forceinline__ const int32_t* formula_terms(const PrepView& v, int32_t off, int32_t q, int dedup, int32_t* nt) {
    const bool uniq = F == Formula::COS || (F == Formula::BM25 && dedup);
    *nt = uniq ? v.u_cnt[q] : v.o_cnt[q];
    return (uniq ? v.u_terms : v.o_terms) + off;
}

template <Formula F>
__device__ __forceinline__ double formula_score(const RescoreIndex& r, const int32_t* terms, int32_t nt, uint32_t doc) {
    if constexpr (F == Formula::BM25) return score_bm25(r, terms, nt, doc);
    else if constexpr (F == Formula::COS) return score_cos(r, terms, nt, doc);
    else return score_v3(r, terms, nt, doc);
}

// Ranges layout, grid-stride over every candidate: query q owns [cand_off[q], cand_off[q+1]) (dense path, explicit
// candidate lists of br_rescore_docs / br_rerank_v3_scores).
template <Formula F>
__global__ void k_rescore(RescoreIndex r, const int32_t* __restrict__ q_off, PrepView v, int dedup,
                          const int64_t* __restrict__ cand_off, int32_t q_begin, int32_t nq,
                          const int32_t* __restrict__ cand, double* __restrict__ cand_score) {
    const int64_t c0 = cand_off[q_begin], c1 = cand_off[q_begin + nq];
    for (int64_t c = c0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < c1; c += (int64_t)gridDim.x * blockDim.x) {
        const int32_t doc = cand[c];
        if (doc < 0) { cand_score[c] = 0.0; continue; }          // empty candidate slot
        int32_t lo = q_begin, hi = q_begin + nq;
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (cand_off[mid] <= c) lo = mid; else hi = mid;
        }
        int32_t nt;
        const int32_t* terms = formula_terms<F>(v, q_off[lo], lo, dedup, &nt);
        cand_score[c] = formula_score<F>(r, terms, nt, (uint32_t)doc);
    }
}

// Stride layout, one CTA per query: query q owns [q*stride, (q+1)*stride), only its first cnt[q] slots are live (tiled
// path, br_fuse_linear's candidate union).
template <Formula F>
__global__ void __launch_bounds__(64) k_rescore_heads(RescoreIndex r, const int32_t* __restrict__ q_off, PrepView v, int dedup,
                                                      int32_t stride, const int32_t* __restrict__ cnt,
                                                      const int32_t* __restrict__ cand, double* __restrict__ cand_score) {
    const int q = blockIdx.x;
    const int n = min(cnt[q], stride);
    int32_t nt;
    const int32_t* terms = formula_terms<F>(v, q_off[q], q, dedup, &nt);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int64_t c = (int64_t)q * stride + i;
        const int32_t doc = cand[c];
        cand_score[c] = doc < 0 ? 0.0 : formula_score<F>(r, terms, nt, (uint32_t)doc);   // 0.0: empty candidate slot
    }
}

// ------------------------------------------------------------------------------------------
// final select: (score desc, id asc), duplicates removed, streaming over any number of candidates
// ------------------------------------------------------------------------------------------
constexpr int FS_T = 256, FS_N = 2048;

struct FsKey {
    double s;
    int64_t id;
};
__device__ __forceinline__ bool fs_before(const FsKey& a, const FsKey& b) {
    return a.s > b.s || (a.s == b.s && a.id < b.id);
}

__device__ void fs_sort(FsKey* keys, int n) {  // bitonic over keys[0, n), n a power of two <= FS_N
    for (int size = 2; size <= n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < n / 2; i += FS_T) {
                const int a = 2 * i - (i & (stride - 1));
                const int b = a + stride;
                const bool up = (a & size) == 0;
                const FsKey ka = keys[a], kb = keys[b];
                if (fs_before(kb, ka) == up) { keys[a] = kb; keys[b] = ka; }
            }
        }
    }
    __syncthreads();
}

// Candidates of query q: parts p = 0..n_parts-1, each the range [off_p, off_p + cnt_p) of ids/scores.
template <class IdT>
__global__ void __launch_bounds__(FS_T) k_final_select(const IdT* __restrict__ ids, const double* __restrict__ sc,
                                                       const int64_t* __restrict__ cand_off, int32_t q_begin,
                                                       int32_t n_parts, int64_t part_stride, int32_t fixed_cnt,
                                                       int32_t k, int64_t id_base, int positive_only,
                                                       IdT* __restrict__ out_ids, double* __restrict__ out_sc,
                                                       int32_t* __restrict__ out_cnt, const int32_t* __restrict__ cnt_hint,
                                                       const br_record* __restrict__ recs = nullptr) {
    __shared__ FsKey keys[FS_N];
    __shared__ uint32_t s_flag[FS_N];
    const int q = q_begin + blockIdx.x;
    const FsKey pad = {-CUDART_INF, INT64_MAX};
    int n_best = 0;  // unique entries currently kept in keys[0, n_best)
    int part = 0;
    int64_t pos = 0;
    bool done = false;
    while (!done) {
        // fill keys[n_best, FS_N) from the candidate stream
        int filled = n_best;
        __syncthreads();
        while (filled < FS_N && part < n_parts) {
            const int64_t base = cand_off ? cand_off[q] : (int64_t)part * part_stride + (int64_t)q * fixed_cnt;
            int64_t cnt = cand_off ? cand_off[q + 1] - cand_off[q] : fixed_cnt;
            if (cnt_hint) cnt = min(cnt, (int64_t)max(cnt_hint[q], 0));      // only the head of the region is in use
            const int64_t take = min((int64_t)(FS_N - filled), cnt - pos);
            for (int64_t i = threadIdx.x; i < take; i += FS_T) {
                IdT id;
                double scv;
                if (recs) { const br_record r = recs[base + pos + i]; id = (IdT)r.id; scv = r.score; }   // packed {id, score}
                else { id = ids[base + pos + i]; scv = sc[base + pos + i]; }
                FsKey kk = {scv, (int64_t)id};
                if (id < 0 || (positive_only && scv == 0.0)) kk = pad;      // positive_only: float64 score != 0 only
                keys[filled + i] = kk;
            }
            filled += (int)take;
            pos += take;
            if (pos >= cnt) { ++part; pos = 0; }
        }
        done = part >= n_parts;
        int n_sort = 64;                                   // smallest power of two covering the filled part
        while (n_sort < filled) n_sort <<= 1;
        for (int i = filled + threadIdx.x; i < FS_N; i += FS_T) keys[i] = pad;
        fs_sort(keys, n_sort);
        // unique-compact the head into keys[0, k)
        for (int i = threadIdx.x; i < FS_N; i += FS_T)
            s_flag[i] = (keys[i].id != INT64_MAX && (i == 0 || keys[i].id != keys[i - 1].id ||
                                                     keys[i].s != keys[i - 1].s)) ? 1u : 0u;
        __syncthreads();
        // exclusive scan of flags over FS_N (FS_N / FS_T per thread, blocked)
        constexpr int PER = FS_N / FS_T;
        uint32_t loc[PER], sum = 0;
#pragma unroll
        for (int j = 0; j < PER; ++j) { loc[j] = s_flag[threadIdx.x * PER + j]; sum += loc[j]; }
        uint32_t total;
        uint32_t ex = block_excl_scan(sum, &total);
        FsKey mine[PER];
#pragma unroll
        for (int j = 0; j < PER; ++j) mine[j] = keys[threadIdx.x * PER + j];
        __syncthreads();
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            if (loc[j]) { if (ex < (uint32_t)k) keys[ex] = mine[j]; ++ex; }
        }
        __syncthreads();
        n_best = (int)min(total, (uint32_t)k);
    }
    for (int i = threadIdx.x; i < k; i += FS_T) {
        const bool valid = i < n_best;
        out_ids[(int64_t)q * k + i] = valid ? (IdT)(keys[i].id + id_base) : (IdT)-1;
        out_sc[(int64_t)q * k + i] = valid ? keys[i].s : 0.0;
    }
    if (out_cnt && threadIdx.x == 0) out_cnt[q] = n_best;
}


// TF-IDF cosine first stage (cosine_similarity_bm25_reranking.py:72-110,121-126,210-226): doc vector tf*idf,
// query vector idf per distinct in-corpus term, both L2-normalised.  cos(d,q) = sum_t (tf*idf_t)*idf_t /
// (||d|| ||q||); ||q|| is constant per query, so ranking needs only w'[d,t] = tf*idf_t^2/||d|| per posting -
// the same packed-posting layout as BM25, scored by the same kernels.
__global__ void k_tfidf_norm2(const int64_t* __restrict__ row_ptr, int32_t vocab, int64_t nnz,
                              const br_posting* __restrict__ post, const uint16_t* __restrict__ tf,
                              const double* __restrict__ idf, double* __restrict__ norm2) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    int32_t lo = 0, hi = vocab;
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (row_ptr[mid] <= j) lo = mid; else hi = mid;
    }
    const double e = (double)(float)((double)tf[j] * idf[lo]);   // stored as float32 in the reference's lil_matrix (:88)
    atomicAdd(norm2 + post[j].doc, e * e);                      // doc_norms are float64 (scipy norm(axis=1), :210)
}
// norm2 -> 1/sqrt(norm2) in place (0 for an empty doc: its cosine row is all zero, SURVEY a11)
__global__ void k_tfidf_invnorm(double* __restrict__ norm2, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) norm2[i] = norm2[i] > 0.0 ? 1.0 / sqrt(norm2[i]) : 0.0;
}
__global__ void k_tfidf_weights(const int64_t* __restrict__ row_ptr, int32_t vocab, int64_t nnz,
                                const br_posting* __restrict__ post, const uint16_t* __restrict__ tf,
                                const double* __restrict__ idf, const double* __restrict__ inv_norm,
                                br_posting* __restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    int32_t lo = 0, hi = vocab;
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (row_ptr[mid] <= j) lo = mid; else hi = mid;
    }
    const uint32_t d = post[j].doc;
    const float e = (float)((double)tf[j] * idf[lo]);
    out[j].doc = d;
    out[j].w = (float)((double)e * (double)(float)idf[lo] * inv_norm[d]);
}

__global__ void k_scatter_rows(const int32_t* __restrict__ rows, int32_t ns, int32_t k, const int32_t* __restrict__ ids,
                               const double* __restrict__ sc, const int32_t* __restrict__ cnt, int32_t* __restrict__ out_ids,
                               double* __restrict__ out_sc, int32_t* __restrict__ out_cnt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)ns * k) return;
    const int32_t r = (int32_t)(i / k), c = (int32_t)(i - (int64_t)r * k);
    const int64_t o = (int64_t)rows[r] * k + c;
    out_ids[o] = ids[i];
    out_sc[o] = sc[i];
    if (c == 0 && out_cnt) out_cnt[rows[r]] = cnt[r];
}

// ------------------------------------------------------------------------------------------
// host drivers
// ------------------------------------------------------------------------------------------

static RescoreIndex rescore_view(const br_index* ix) {
    return RescoreIndex{ix->post, ix->tf, ix->row_ptr, ix->dl, ix->idf, ix->cos_inv_norm, ix->hot_slot, ix->skip, ix->n_sub,
                        ix->sub_shift, ix->avgdl, ix->k1, ix->b, ix->variant};
}

int launch_rescore(br_index* ix, Formula f, const int32_t* q_off, const PrepView& pv, int dedup, const int64_t* cand_off,
                   int32_t q_begin, int32_t nq, const int32_t* cand, double* cand_score, int64_t total, cudaStream_t st) {
    const int64_t blocks = total < 0 ? kNumSMs * 16 : std::max<int64_t>(1, std::min<int64_t>((total + 127) / 128, kNumSMs * 16));
    auto* kern = f == Formula::BM25 ? &k_rescore<Formula::BM25> : f == Formula::COS ? &k_rescore<Formula::COS> : &k_rescore<Formula::V3>;
    kern<<<(unsigned)blocks, 128, 0, st>>>(rescore_view(ix), q_off, pv, dedup, cand_off, q_begin, nq, cand, cand_score);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

int launch_rescore_heads(br_index* ix, Formula f, const int32_t* q_off, const PrepView& pv, int dedup, int32_t nq,
                         int32_t stride, const int32_t* cnt, const int32_t* cand, double* cand_score, cudaStream_t st) {
    auto* kern = f == Formula::BM25 ? &k_rescore_heads<Formula::BM25>
               : f == Formula::COS  ? &k_rescore_heads<Formula::COS> : &k_rescore_heads<Formula::V3>;
    kern<<<nq, 64, 0, st>>>(rescore_view(ix), q_off, pv, dedup, stride, cnt, cand, cand_score);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

int launch_final_select(const int32_t* cand, const double* cand_score, const int64_t* cand_off, int32_t q_begin,
                        int32_t nq, int32_t k, int positive_only, int32_t* out_ids, double* out_scores,
                        int32_t* out_counts, cudaStream_t st, const int32_t* cnt_hint, int32_t fixed_cnt) {
    k_final_select<int32_t><<<nq, FS_T, 0, st>>>(cand, cand_score, cand_off, q_begin, 1, 0, fixed_cnt, k, 0, positive_only,
                                                 out_ids, out_scores, out_counts, cnt_hint);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}
// n_terms >= 0: the caller knows q_offsets[nq] (or an upper bound) - no device read, no stream synchronisation.
int prep_queries(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int dedup, cudaStream_t st,
                 PrepView* pv, int64_t** chunk_start, int32_t n_terms) {
    int32_t T = n_terms;
    if (T < 0) {
        BR_CUDA(cudaMemcpyAsync(&T, q_off + nq, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaStreamSynchronize(st));
    }
    BR_REQUIRE(T >= 0, BR_ERR_INVALID, "query offsets: negative total");
    const size_t Tn = (size_t)T + 1, Q = (size_t)nq + 2;
    // carve ws_prep
    size_t bytes = 0;
    auto carve = [&](size_t n) { size_t o = bytes; bytes += (n + 255) & ~(size_t)255; return o; };
    const size_t o_ut = carve(Tn * 4), o_um = carve(Tn * 4), o_uc = carve(Tn * 8), o_un = carve(Q * 4),
                 o_ot = carve(Tn * 4), o_on = carve(Q * 4), o_P = carve(Q * 8), o_nc = carve(Q * 4),
                 o_tmp = carve(Tn * 4), o_cs = carve(Q * 8), o_sig = carve(Q * 4), o_sl = carve(Q * 4), o_bad = carve(16);
    BR_TRY(ix->ws_prep.reserve(bytes));
    char* p = ix->ws_prep.as<char>();
    pv->u_terms = (int32_t*)(p + o_ut); pv->u_mult = (int32_t*)(p + o_um); pv->u_cum = (int64_t*)(p + o_uc);
    pv->u_cnt = (int32_t*)(p + o_un); pv->o_terms = (int32_t*)(p + o_ot); pv->o_cnt = (int32_t*)(p + o_on);
    pv->P = (int64_t*)(p + o_P); pv->n_chunks = (uint32_t*)(p + o_nc); pv->tmp = (int32_t*)(p + o_tmp); pv->sig = (uint32_t*)(p + o_sig);
    pv->slack = (float*)(p + o_sl);
    *chunk_start = (int64_t*)(p + o_cs);
    pv->t_cap = T;
    pv->bad = (int32_t*)(p + o_bad);
    BR_CUDA(cudaMemsetAsync(pv->bad, 0, 4, st));
    k_prep_queries<<<blocks_for((int64_t)nq * 32, 128), 128, 0, st>>>(q_terms, q_off, nq, ix->vocab, ix->row_ptr, ix->sig_bit, dedup,
                                                                    ix->idf, ix->amax, *pv);
    BR_CUDA(cudaGetLastError());
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(pv->n_chunks, nq, *chunk_start);
    BR_CUDA(cudaGetLastError());
    ix->stats.kernel_launches += 2;
    return BR_OK;
}

int score_batch(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int dedup, float* out,
                cudaStream_t st) {
    BR_REQUIRE(ix && q_terms && q_off && out, BR_ERR_INVALID, "br_score_batch: null pointer");
    BR_REQUIRE(ix->finalized, BR_ERR_STATE, "br_score_batch: call br_index_finalize first");
    BR_REQUIRE(nq >= 0, BR_ERR_INVALID, "br_score_batch: nq < 0");
    if (nq == 0) return BR_OK;
    BR_CUDA(cudaSetDevice(ix->device));
    ix->stats = br_query_stats{};
    PrepView pv;
    int64_t* chunk_start;
    BR_TRY(prep_queries(ix, q_terms, q_off, nq, dedup, st, &pv, &chunk_start));
    BR_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)nq * (size_t)ix->n_docs, st));
    k_score_dense<<<kNumSMs * 8, 256, 0, st>>>(ix->post, ix->row_ptr, q_off, pv, chunk_start, 0, nq, out, ix->n_docs,
                                               HitRows{});
    BR_CUDA(cudaGetLastError());
    ix->stats.kernel_launches += 1;
    ix->stats.queries_dense += nq;
    return BR_OK;
}

// Dense path for queries [q_begin, q_begin + nq) of a prepared batch; results into out_* rows.
static int topk_dense(br_index* ix, const int32_t* q_off, const PrepView& pv, const int64_t* chunk_start,
                      int32_t q_begin, int32_t nq, int32_t k, int dedup, int positive_only, int32_t* out_ids,
                      double* out_scores, int32_t* out_counts, cudaStream_t st, const br_posting* post_table = nullptr,
                      const DocFilter* filt = nullptr) {
    // post_table != nullptr: score with that weight table (TF-IDF cosine stage) and re-score the candidate band with the
    // float64 cosine; otherwise BM25 weights + exact float64 BM25 re-score of the band.
    const Formula formula = post_table ? Formula::COS : Formula::BM25;
    const br_posting* post = post_table ? post_table : ix->post;
    const DocFilter f = filt ? *filt : DocFilter{};
    const int64_t N = ix->n_docs;
    // queries per pass: dense fp32 rows within ~1 GiB
    int32_t qb = (int32_t)std::max<int64_t>(1, std::min<int64_t>(nq, (1LL << 30) / (4 * N)));
    // BM25 under okapi_no_plus1: a hit row per query (used only by the queries with a term of negative idf) after the
    // fp32 rows, 1/32 of their size
    const bool mixed = !post_table && ix->amax;
    const size_t dense_bytes = (sizeof(float) * (size_t)qb * (size_t)N + 255) & ~(size_t)255;
    HitRows hits{};
    hits.words = (N + 31) / 32;
    BR_TRY(ix->ws_dense.reserve(dense_bytes + (mixed ? sizeof(uint32_t) * (size_t)qb * (size_t)hits.words : 0)));
    float* dense = ix->ws_dense.as<float>();
    if (mixed) {
        hits.slack = pv.slack;
        hits.bits = (uint32_t*)(ix->ws_dense.as<char>() + dense_bytes);
    }
    // selection scratch for the whole batch slice
    size_t bytes = 0;
    auto carve = [&](size_t n) { size_t o = bytes; bytes += (n + 255) & ~(size_t)255; return o; };
    const size_t Q = (size_t)(q_begin + nq) + 2;
    const size_t o_lo = carve(Q * 4), o_mode = carve(Q * 4), o_z = carve(Q * 4), o_cnt = carve(Q * 8), o_off = carve(Q * 8);
    BR_TRY(ix->ws_sel.reserve(bytes));
    char* p = ix->ws_sel.as<char>();
    SelView sv{(float*)(p + o_lo), (int32_t*)(p + o_mode), (int32_t*)(p + o_z), (int64_t*)(p + o_cnt)};
    int64_t* cand_off = (int64_t*)(p + o_off);
    std::vector<int64_t> h_cnt((size_t)qb), h_off((size_t)qb + 1);
    for (int32_t s = 0; s < nq; s += qb) {
        const int32_t b0 = q_begin + s, bn = std::min(qb, nq - s);
        BR_CUDA(cudaMemsetAsync(dense, 0, sizeof(float) * (size_t)bn * (size_t)N, st));
        if (mixed) BR_CUDA(cudaMemsetAsync(hits.bits, 0, sizeof(uint32_t) * (size_t)bn * (size_t)hits.words, st));
        ix->prof_begin(st);
        k_score_dense<<<kNumSMs * 8, 256, 0, st>>>(post, ix->row_ptr, q_off, pv, chunk_start, b0, bn, dense, N, hits);
        BR_CUDA(cudaGetLastError());
        ix->prof_end(st);
        // (query chunks keep batch-wide query indices b0 + i, so the filter rows need no remapping here)
        k_select_radix<<<bn, SEL_T, 0, st>>>(dense, N, k, positive_only, sv, b0, dedup ? pv.u_cnt : pv.o_cnt, f, hits);
        BR_CUDA(cudaGetLastError());
        BR_CUDA(cudaMemcpyAsync(h_cnt.data(), sv.cnt + b0, sizeof(int64_t) * (size_t)bn, cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaStreamSynchronize(st));
        int64_t total = 0;
        for (int32_t i = 0; i < bn; ++i) { h_off[(size_t)i] = total; total += h_cnt[(size_t)i]; }
        h_off[(size_t)bn] = total;
        BR_CUDA(cudaMemcpyAsync(cand_off + b0, h_off.data(), sizeof(int64_t) * ((size_t)bn + 1), cudaMemcpyHostToDevice, st));
        BR_TRY(ix->ws_cand.reserve((size_t)(total + 1) * (sizeof(int32_t) + sizeof(double)) + 256));
        int32_t* cand = ix->ws_cand.as<int32_t>();
        double* cand_sc = (double*)(ix->ws_cand.as<char>() + (((size_t)(total + 1) * sizeof(int32_t) + 255) & ~(size_t)255));
        k_emit_cands<<<bn, SEL_T, 0, st>>>(dense, N, positive_only, sv, b0, cand_off, cand, f, hits);
        BR_CUDA(cudaGetLastError());
        if (total > 0) BR_TRY(launch_rescore(ix, formula, q_off, pv, dedup, cand_off, b0, bn, cand, cand_sc, total, st));
        BR_TRY(launch_final_select(cand, cand_sc, cand_off, b0, bn, k, positive_only, out_ids, out_scores, out_counts, st));
        // cand_off/h_off are reused by the next pass
        BR_CUDA(cudaStreamSynchronize(st));
        ix->stats.kernel_launches += 5;
        ix->stats.candidates_rescored += total;
    }
    ix->stats.queries_dense += nq;
    return BR_OK;
}

// (local id, score) -> {global id, score} records, the unit of the cross-shard all-gather
__global__ void k_pack_records(const int32_t* __restrict__ ids, const double* __restrict__ sc, int64_t n, int64_t doc_base,
                               br_record* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t d = ids[i];
    out[i] = br_record{d >= 0 ? (int64_t)d + doc_base : (int64_t)-1, sc[i]};
}

int check_doc_filter(const br_doc_filter* filter, int64_t n_ids, const char* ids, const std::string& fn) {
    if (!filter) return BR_OK;
    BR_REQUIRE(filter->bits_dev, BR_ERR_INVALID, fn + ": filter bitmap is null");
    BR_REQUIRE(filter->n_rows >= 1, BR_ERR_INVALID, fn + ": filter n_rows must be >= 1");
    BR_REQUIRE(filter->words >= (n_ids + 31) / 32, BR_ERR_INVALID, fn + ": filter words < ceil(" + ids + " / 32)");
    return BR_OK;
}

// *bad is reported when the call returns; the -1 for a bad value means no kernel ever addresses a row that does not exist.
__global__ void k_filter_rows(const int32_t* __restrict__ in, int32_t nq, int32_t n_rows, int32_t* __restrict__ out,
                              int32_t* __restrict__ bad) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const int32_t r = in ? in[q] : 0;
    const bool ok = r >= -1 && r < n_rows;
    if (!ok) atomicOr(bad, 1);
    out[q] = ok ? r : -1;
}
// filter rows of a compacted sub-batch: out[i] = in[idx[i]]
__global__ void k_gather_rows(const int32_t* __restrict__ idx, int32_t n, const int32_t* __restrict__ in, int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[idx[i]];
}

// A prepared batch through the tiled path, then - for the queries it cannot serve exactly - the long-query pass and the
// dense path.  post_table: weight table of the TF-IDF cosine stage (nullptr: BM25).  filt: the batch's doc filter
// (nullptr: none); sub_rows: int32[nq] scratch for the filter rows of the compacted sub-batches.
static int serve_prepared(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int32_t k, int dedup,
                          int positive_only, const PrepView& pv, const int64_t* chunk_start, int32_t* out_ids,
                          double* out_scores, int32_t* out_counts, cudaStream_t st, const br_posting* post_table,
                          const DocFilter* filt = nullptr, int32_t* sub_rows = nullptr) {
    if (!fused_supported(ix, k, nq, post_table != nullptr)) {
        BR_TRY(topk_dense(ix, q_off, pv, chunk_start, 0, nq, k, dedup, positive_only, out_ids, out_scores, out_counts, st, post_table,
                          filt));
    } else {
        std::vector<int32_t> flags;
        BR_TRY(topk_fused(ix, q_off, pv, nq, k, dedup, positive_only, out_ids, out_scores, out_counts, st, &flags, false, post_table,
                          filt));
        {   // offsets past n_terms make queries empty: report before the scratch of this batch is reused below
            int32_t h_bad = 0;
            BR_CUDA(cudaMemcpyAsync(&h_bad, pv.bad, 4, cudaMemcpyDeviceToHost, st));
            BR_CUDA(cudaStreamSynchronize(st));
            BR_REQUIRE(!h_bad, BR_ERR_INVALID, "br_topk_batch: q_offsets run past n_terms");
        }
        std::vector<int32_t> redo;
        for (int32_t q = 0; q < nq; ++q) if (flags[(size_t)q]) redo.push_back(q);
        ix->stats.queries_fused += nq - (int64_t)redo.size();
        if (!redo.empty()) {
            // The queries the regular pass cannot serve exactly (more than 32 terms / 20 hot terms, candidate overflow,
            // fewer than k docs with a hit) are compacted into a sub-batch: first the long-query pass of the tiled
            // scorer (up to 64 terms / 40 hot terms: bigram-expanded queries), then, for what is still left, the dense path.
            // n_terms may be an upper bound of q_offsets[nq]: copy the batch's own terms only (q_offsets[nq] <= n_terms
            // was checked above)
            std::vector<int32_t> h_off((size_t)nq + 1);
            BR_CUDA(cudaMemcpyAsync(h_off.data(), q_off, 4 * ((size_t)nq + 1), cudaMemcpyDeviceToHost, st));
            BR_CUDA(cudaStreamSynchronize(st));
            std::vector<int32_t> h_terms((size_t)h_off[(size_t)nq]);
            BR_CUDA(cudaMemcpyAsync(h_terms.data(), q_terms, 4 * h_terms.size(), cudaMemcpyDeviceToHost, st));
            BR_CUDA(cudaStreamSynchronize(st));
            for (int pass = 0; pass < 2 && !redo.empty(); ++pass) {
                const bool long_pass = pass == 0;
                if (long_pass && !ix->allow_fused_long) continue;
                const int32_t ns = (int32_t)redo.size();
                std::vector<int32_t> s_off((size_t)ns + 1, 0), s_terms;
                for (int32_t i = 0; i < ns; ++i) {
                    const int32_t q = redo[(size_t)i];
                    s_terms.insert(s_terms.end(), h_terms.begin() + h_off[(size_t)q], h_terms.begin() + h_off[(size_t)q + 1]);
                    s_off[(size_t)i + 1] = (int32_t)s_terms.size();
                }
                size_t bytes = 0;
                auto carve = [&](size_t n) { size_t o = bytes; bytes += (n + 255) & ~(size_t)255; return o; };
                const size_t o_t = carve(4 * (s_terms.size() + 1)), o_o = carve(4 * ((size_t)ns + 1)), o_q = carve(4 * (size_t)ns),
                             o_i = carve(4 * (size_t)ns * k), o_s = carve(8 * (size_t)ns * k), o_c = carve(4 * (size_t)ns);
                BR_TRY(ix->ws_misc.reserve(bytes));
                char* p = ix->ws_misc.as<char>();
                int32_t *d_t = (int32_t*)(p + o_t), *d_o = (int32_t*)(p + o_o), *d_q = (int32_t*)(p + o_q),
                        *d_i = (int32_t*)(p + o_i), *d_c = (int32_t*)(p + o_c);
                double* d_s = (double*)(p + o_s);
                BR_CUDA(cudaMemcpyAsync(d_t, s_terms.data(), 4 * s_terms.size(), cudaMemcpyHostToDevice, st));
                BR_CUDA(cudaMemcpyAsync(d_o, s_off.data(), 4 * ((size_t)ns + 1), cudaMemcpyHostToDevice, st));
                BR_CUDA(cudaMemcpyAsync(d_q, redo.data(), 4 * (size_t)ns, cudaMemcpyHostToDevice, st));
                // sub-batch query i is batch query redo[i]: its filter row is the batch's row of redo[i]
                DocFilter sfilt{};
                if (filt) {
                    sfilt = *filt;
                    sfilt.row = sub_rows;
                    k_gather_rows<<<blocks_for(ns, 256), 256, 0, st>>>(d_q, ns, filt->row, sub_rows);
                    BR_CUDA(cudaGetLastError());
                    ix->stats.kernel_launches += 1;
                }
                const DocFilter* sf = filt ? &sfilt : nullptr;
                PrepView spv;
                int64_t* s_chunk;
                BR_TRY(prep_queries(ix, d_t, d_o, ns, dedup, st, &spv, &s_chunk, (int32_t)s_terms.size()));
                std::vector<int32_t> next;
                if (long_pass) {
                    std::vector<int32_t> f2;
                    BR_TRY(topk_fused(ix, d_o, spv, ns, k, dedup, positive_only, d_i, d_s, d_c, st, &f2, true, post_table, sf));
                    for (int32_t i = 0; i < ns; ++i) if (f2[(size_t)i]) next.push_back(redo[(size_t)i]);
                    ix->stats.queries_fused += ns - (int64_t)next.size();
                } else {
                    BR_TRY(topk_dense(ix, d_o, spv, s_chunk, 0, ns, k, dedup, positive_only, d_i, d_s, d_c, st, post_table, sf));
                }
                // rows of queries that go on to the next pass are overwritten there (same stream)
                k_scatter_rows<<<blocks_for((int64_t)ns * k, 256), 256, 0, st>>>(d_q, ns, k, d_i, d_s, d_c, out_ids, out_scores,
                                                                                out_counts);
                BR_CUDA(cudaGetLastError());
                BR_CUDA(cudaStreamSynchronize(st));              // the host vectors and ws_misc are reused by the next pass
                ix->stats.kernel_launches += 1;
                redo.swap(next);
            }
        }
    }
    return BR_OK;
}

int topk_batch(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int32_t n_terms, int32_t k, int dedup,
               int positive_only, int32_t* out_ids, double* out_scores, int32_t* out_counts, br_record* out_recs,
               const br_doc_filter* filter, cudaStream_t st) {
    BR_REQUIRE(ix && q_terms && q_off && ((out_ids && out_scores) || out_recs), BR_ERR_INVALID, "br_topk_batch: null pointer");
    BR_REQUIRE(ix->finalized, BR_ERR_STATE, "br_topk_batch: call br_index_finalize first");
    BR_REQUIRE(k >= 1 && k <= BR_MAX_K, BR_ERR_INVALID, "br_topk_batch: k must be in [1, BR_MAX_K]");
    BR_REQUIRE(nq >= 0, BR_ERR_INVALID, "br_topk_batch: nq < 0");
    BR_TRY(check_doc_filter(filter, ix->n_docs, "n_docs", "br_topk_batch"));
    if (nq == 0) return BR_OK;
    BR_CUDA(cudaSetDevice(ix->device));
    ix->stats = br_query_stats{};
    // filter rows: [nq] of the batch, [nq] of its redo sub-batches, the device-side "bad row" flag
    DocFilter fv{};
    const DocFilter* filt = nullptr;
    int32_t* f_sub = nullptr;
    int32_t* f_bad = nullptr;
    if (filter) {
        const size_t rb = ((size_t)nq * 4 + 255) & ~(size_t)255;
        BR_TRY(ix->ws_filt.reserve(2 * rb + 256));
        char* fp = ix->ws_filt.as<char>();
        int32_t* rows = (int32_t*)fp;
        f_sub = (int32_t*)(fp + rb);
        f_bad = (int32_t*)(fp + 2 * rb);
        BR_CUDA(cudaMemsetAsync(f_bad, 0, 4, st));
        k_filter_rows<<<blocks_for(nq, 256), 256, 0, st>>>(filter->query_row_dev, nq, filter->n_rows, rows, f_bad);
        BR_CUDA(cudaGetLastError());
        ix->stats.kernel_launches += 1;
        fv = DocFilter{filter->bits_dev, filter->words, rows};
        filt = &fv;
    }
    if (!out_ids || !out_scores) {                         // records only: ids / scores go to scratch
        BR_TRY(ix->ws_rec.reserve((size_t)nq * k * 12 + 512));
        out_ids = ix->ws_rec.as<int32_t>();
        out_scores = (double*)(ix->ws_rec.as<char>() + (((size_t)nq * k * 4 + 255) & ~(size_t)255));
    }
    PrepView pv;
    int64_t* chunk_start;
    BR_TRY(prep_queries(ix, q_terms, q_off, nq, dedup, st, &pv, &chunk_start, n_terms));
    // algorithmic bytes of this batch: 8 B per posting of every distinct in-vocab query term
    std::vector<int64_t> hP((size_t)nq);
    BR_CUDA(cudaMemcpyAsync(hP.data(), pv.P, sizeof(int64_t) * (size_t)nq, cudaMemcpyDeviceToHost, st));
    BR_TRY(serve_prepared(ix, q_terms, q_off, nq, k, dedup, positive_only, pv, chunk_start, out_ids, out_scores, out_counts, st,
                          nullptr, filt, f_sub));
    if (out_recs) {
        k_pack_records<<<blocks_for((int64_t)nq * k, 256), 256, 0, st>>>(out_ids, out_scores, (int64_t)nq * k, ix->doc_base, out_recs);
        BR_CUDA(cudaGetLastError());
        ix->stats.kernel_launches += 1;
    }
    int32_t h_fbad = 0;
    if (f_bad) BR_CUDA(cudaMemcpyAsync(&h_fbad, f_bad, 4, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    int64_t sum = 0;
    for (int64_t v : hP) sum += v;
    ix->stats.postings_bytes = 8 * sum;
    ix->prof_collect();
    BR_REQUIRE(!h_fbad, BR_ERR_INVALID, "br_topk_batch: a filter query_row is outside [-1, n_rows)");
    return BR_OK;
}

int rescore_docs(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int dedup,
                 const int32_t* cand_ids, const int64_t* cand_off, double* out_scores, cudaStream_t st) {
    BR_REQUIRE(ix && q_terms && q_off && cand_ids && cand_off && out_scores, BR_ERR_INVALID, "br_rescore_docs: null pointer");
    BR_REQUIRE(ix->finalized, BR_ERR_STATE, "br_rescore_docs: call br_index_finalize first");
    if (nq <= 0) return BR_OK;
    BR_CUDA(cudaSetDevice(ix->device));
    PrepView pv;
    int64_t* chunk_start;
    BR_TRY(prep_queries(ix, q_terms, q_off, nq, dedup, st, &pv, &chunk_start));
    return launch_rescore(ix, Formula::BM25, q_off, pv, dedup, cand_off, 0, nq, cand_ids, out_scores, -1, st);
}

int enable_tfidf(br_index* ix, cudaStream_t st) {
    BR_REQUIRE(ix && ix->finalized, BR_ERR_STATE, "br_index_enable_tfidf: call br_index_finalize first");
    if (ix->post_cos) return BR_OK;
    BR_CUDA(cudaSetDevice(ix->device));
    DevArray<double> inv_norm;               // owned by the index only once both allocations succeed
    DevArray<br_posting> post_cos;
    BR_TRY(inv_norm.alloc((size_t)ix->n_docs));
    BR_TRY(post_cos.alloc((size_t)ix->nnz));
    ix->cos_inv_norm = std::move(inv_norm);
    ix->post_cos = std::move(post_cos);
    BR_CUDA(cudaMemsetAsync(ix->cos_inv_norm, 0, sizeof(double) * (size_t)ix->n_docs, st));
    if (ix->nnz > 0) {
        k_tfidf_norm2<<<blocks_for(ix->nnz, 256), 256, 0, st>>>(ix->row_ptr, ix->vocab, ix->nnz, ix->post, ix->tf, ix->idf,
                                                                ix->cos_inv_norm);
        k_tfidf_invnorm<<<blocks_for(ix->n_docs, 256), 256, 0, st>>>(ix->cos_inv_norm, ix->n_docs);
        k_tfidf_weights<<<blocks_for(ix->nnz, 256), 256, 0, st>>>(ix->row_ptr, ix->vocab, ix->nnz, ix->post, ix->tf, ix->idf,
                                                                  ix->cos_inv_norm, ix->post_cos);
    }
    BR_CUDA(cudaStreamSynchronize(st));
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

int tfidf_topk(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int32_t k, int32_t* out_ids,
               double* out_scores, int32_t* out_counts, cudaStream_t st) {
    BR_REQUIRE(ix && q_terms && q_off && out_ids && out_scores, BR_ERR_INVALID, "br_tfidf_cosine_topk: null pointer");
    BR_REQUIRE(k >= 1 && k <= BR_MAX_K && nq >= 0, BR_ERR_INVALID, "br_tfidf_cosine_topk: bad sizes");
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_tfidf_cosine_topk: null handle");
    BR_CUDA(cudaSetDevice(ix->device));
    BR_TRY(enable_tfidf(ix, st));
    if (nq == 0) return BR_OK;
    ix->stats = br_query_stats{};
    PrepView pv;
    int64_t* chunk_start;
    BR_TRY(prep_queries(ix, q_terms, q_off, nq, 1 /* binary query tf: generate_query_embedding sets, not adds */, st, &pv,
                        &chunk_start));
    // same tiled scorer as BM25 over the tf*idf^2/||d|| table (round 2 ran this stage on the dense scatter-add path)
    BR_TRY(serve_prepared(ix, q_terms, q_off, nq, k, 1, 0, pv, chunk_start, out_ids, out_scores, out_counts, st, ix->post_cos));
    BR_CUDA(cudaStreamSynchronize(st));
    ix->prof_collect();
    return BR_OK;
}

int rerank_v3(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, const int32_t* cand_ids,
              const int64_t* cand_off, double* out_scores, cudaStream_t st) {
    BR_REQUIRE(ix && q_terms && q_off && cand_ids && cand_off && out_scores, BR_ERR_INVALID, "br_rerank_v3_scores: null pointer");
    BR_REQUIRE(ix->finalized, BR_ERR_STATE, "br_rerank_v3_scores: call br_index_finalize first");
    if (nq <= 0) return BR_OK;
    BR_CUDA(cudaSetDevice(ix->device));
    PrepView pv;
    int64_t* chunk_start;
    BR_TRY(prep_queries(ix, q_terms, q_off, nq, 0, st, &pv, &chunk_start));
    return launch_rescore(ix, Formula::V3, q_off, pv, 0, cand_off, 0, nq, cand_ids, out_scores, -1, st);
}

int topk_merge(const int64_t* ids, const double* scores, int32_t n_parts, int32_t nq, int32_t k, int64_t* out_ids,
               double* out_scores, cudaStream_t st) {
    BR_REQUIRE(ids && scores && out_ids && out_scores, BR_ERR_INVALID, "br_topk_merge: null pointer");
    BR_REQUIRE(n_parts >= 1 && nq >= 0 && k >= 1 && k <= BR_MAX_K, BR_ERR_INVALID, "br_topk_merge: bad sizes");
    if (nq == 0) return BR_OK;
    k_final_select<int64_t><<<nq, FS_T, 0, st>>>(ids, scores, nullptr, 0, n_parts, (int64_t)nq * k, k, k, 0, 0, out_ids,
                                                 out_scores, nullptr, nullptr);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

int topk_merge_records(const br_record* recs, int32_t n_parts, int32_t nq, int32_t k, int64_t* out_ids, double* out_scores,
                       cudaStream_t st) {
    BR_REQUIRE(recs && out_ids && out_scores, BR_ERR_INVALID, "br_topk_merge_records: null pointer");
    BR_REQUIRE(n_parts >= 1 && nq >= 0 && k >= 1 && k <= BR_MAX_K, BR_ERR_INVALID, "br_topk_merge_records: bad sizes");
    if (nq == 0) return BR_OK;
    k_final_select<int64_t><<<nq, FS_T, 0, st>>>(nullptr, nullptr, nullptr, 0, n_parts, (int64_t)nq * k, k, k, 0, 0, out_ids,
                                                 out_scores, nullptr, nullptr, recs);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

}  // namespace br
