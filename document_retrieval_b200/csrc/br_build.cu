// br_build.cu - index build on the GPU: tokenised docs -> CSR posting lists with packed
// (doc id, fp32 BM25 weight) postings, raw tf, dl, df, idf and the hot-term skip tables.
//
// Replaces BM25.__init__/build (bm25_ranking.ipynb:167-189), compute_tf_df_and_avgdl
// (cosine_similarity_bm25_reranking.py:129-172) and build_inverted_index (team_run1.py:80-99).
//
// Pipeline (all on one stream):
//   k_make_keys      one warp per doc: (key = term, value = doc) pairs, dl[doc]       (4 B in, 8 B out / token)
//   radix sort       stable, (term, doc) pairs by the significant bits of the term only - the input is in doc order, so
//                    docs stay ascending inside a term (CUB DeviceRadixSort::SortPairs - library plumbing)
//   k_rle_count/emit run-length encode equal keys -> one posting per (term, doc) with tf = run length
//   k_finish         tf (u16), first/last posting of every term -> df histogram
//   k_exscan         exclusive prefix-scan of df -> row_ptr
//   [host]           idf[t] = log(..) in float64 with libm (bit-identical to math.log)
//   k_weights        w = fp32(idf * ((tf*(k1+1)) / (tf + k1*norm(dl))))  evaluated in float64, no FMA
//   k_skip           per hot term: offset of the first posting of every 2^sub_shift-doc sub-range
//
// Append (br_index_append): the new docs go through the same pipeline as a build of their own, then
//   k_append_rows    row_ptr / df of the grown index (old + new part, per term)
//   k_append_merge   thread per output posting: a term's old postings, then its new ones with doc + N_old  (10 B in, 10 B out)
//
// Remove (br_index_remove): one order-preserving stream compaction of the docs, then of the postings (no term search:
// the CSR is term-major with docs ascending inside a term, and dropping postings keeps that order)
//   k_docmap_count   kept docs per 2048-doc tile, sum(dl) of the kept docs (integer atomics: exact)
//   k_exscan         -> first new id of every tile
//   k_docmap_emit    new_id[doc] = rank among the kept docs (~0u = removed), compacted dl
//   k_remove_count   surviving postings per 2048-posting tile                                  (8 B in + new_id gather)
//   k_exscan         -> first output posting of every tile
//   k_remove_emit    survivors as {new_id[doc], 0.f} + tf; row_ptr of the terms whose rows start in the tile, from the
//                    tile's own ballots                                           (10 B in, 10 B out per kept posting)
//   k_remove_df      df = diff(row_ptr)
#include <math.h>

#include <algorithm>
#include <memory>
#include <thread>

#include <cub/device/device_radix_sort.cuh>

#include "br_common.cuh"
#include "br_kernels.cuh"

namespace br {

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
__global__ void k_make_keys(const int32_t* __restrict__ tok, const int64_t* __restrict__ doc_off,
                            int64_t n_docs, int32_t vocab, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals,
                            uint32_t* __restrict__ dl, int* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t d = warp; d < n_docs; d += n_warps) {
        const int64_t lo = doc_off[d], hi = doc_off[d + 1];
        if (hi < lo || hi - lo > 0xffffffffLL) {
            if (lane == 0) atomicOr(bad, 2);
            continue;
        }
        if (lane == 0) dl[d] = (uint32_t)(hi - lo);
        for (int64_t i = lo + lane; i < hi; i += 32) {
            const int32_t t = tok[i];
            if ((uint32_t)t >= (uint32_t)vocab) atomicOr(bad, 1);
            keys[i] = (uint32_t)t;
            vals[i] = (uint32_t)d;
        }
    }
}

constexpr int RLE_T = 256, RLE_I = 8, RLE_TILE = RLE_T * RLE_I;

__global__ void __launch_bounds__(RLE_T) k_rle_count(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                     int64_t n, uint32_t* __restrict__ block_counts) {
    const int64_t base = (int64_t)blockIdx.x * RLE_TILE;
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < RLE_I; ++j) {
        const int64_t i = base + j * RLE_T + threadIdx.x;   // striped: coalesced, order irrelevant
        if (i < n) c += (i == 0 || keys[i] != keys[i - 1] || vals[i] != vals[i - 1]) ? 1u : 0u;
    }
    uint32_t total;
    block_excl_scan(c, &total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(RLE_T) k_rle_emit(const uint32_t* __restrict__ keys, const uint32_t* __restrict__ vals,
                                                    int64_t n, const int64_t* __restrict__ block_off,
                                                    br_posting* __restrict__ post,
                                                    uint32_t* __restrict__ post_term,
                                                    uint32_t* __restrict__ head_pos) {
    const int64_t base = (int64_t)blockIdx.x * RLE_TILE + (int64_t)threadIdx.x * RLE_I;  // blocked: ordered
    uint64_t k[RLE_I];
    uint64_t prev = (base > 0 && base - 1 < n) ? (((uint64_t)keys[base - 1] << 32) | vals[base - 1]) : ~0ull;
    uint32_t c = 0;
    bool head[RLE_I];
#pragma unroll
    for (int j = 0; j < RLE_I; ++j) {
        const int64_t i = base + j;
        k[j] = i < n ? (((uint64_t)keys[i] << 32) | vals[i]) : 0;
        head[j] = i < n && (i == 0 || k[j] != prev);
        prev = k[j];
        c += head[j] ? 1u : 0u;
    }
    uint32_t total;
    uint32_t ex = block_excl_scan(c, &total);
    int64_t o = block_off[blockIdx.x] + ex;
#pragma unroll
    for (int j = 0; j < RLE_I; ++j) {
        if (head[j]) {
            post[o].doc = (uint32_t)k[j];
            post_term[o] = (uint32_t)(k[j] >> 32);
            head_pos[o] = (uint32_t)(base + j);
            ++o;
        }
    }
}

__global__ void k_finish(const uint32_t* __restrict__ post_term, const uint32_t* __restrict__ head_pos,
                         int64_t nnz, uint32_t n_tokens, uint16_t* __restrict__ tf,
                         uint32_t* __restrict__ tstart, uint32_t* __restrict__ tend, int* __restrict__ bad) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    const uint32_t nxt = j + 1 < nnz ? head_pos[j + 1] : n_tokens;
    const uint32_t f = nxt - head_pos[j];
    if (f > 65535u) atomicOr(bad, 4);
    tf[j] = (uint16_t)f;
    const uint32_t t = post_term[j];
    if (j == 0 || post_term[j - 1] != t) tstart[t] = (uint32_t)j;
    if (j + 1 == nnz || post_term[j + 1] != t) tend[t] = (uint32_t)(j + 1);
}

__global__ void k_df(const uint32_t* __restrict__ tstart, const uint32_t* __restrict__ tend, int32_t vocab,
                     uint32_t* __restrict__ df) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < vocab) df[t] = tend[t] - tstart[t];
}

// Term of posting j = blockIdx.x * blockDim.x + threadIdx.x: the last t with row_ptr[t] <= j, -1 for j >= nnz.  Every
// lane of the warp must call.  The 32 postings of a warp are consecutive, so their terms lie between the term of the
// warp's first and last posting: two full binary searches per warp, the other lanes search only that (mostly one-term)
// range.
__device__ __forceinline__ int32_t warp_term_of(const int64_t* __restrict__ row_ptr, int32_t vocab, int64_t nnz,
                                                int64_t j, int lane) {
    const int64_t j_first = min(j - lane, nnz - 1), j_last = min(j - lane + 31, nnz - 1);
    int32_t t_first = 0, t_last = 0;
    if (j_first >= 0 && (lane == 0 || lane == 31)) {
        const int64_t jj = lane == 0 ? j_first : j_last;
        int32_t a = 0, b = vocab;
        while (b - a > 1) {
            const int32_t mid = (a + b) >> 1;
            if (row_ptr[mid] <= jj) a = mid; else b = mid;
        }
        t_first = t_last = a;
    }
    t_first = __shfl_sync(0xffffffffu, t_first, 0);
    t_last = __shfl_sync(0xffffffffu, t_last, 31);
    if (j >= nnz) return -1;
    int32_t lo = t_first, hi = t_last + 1;  // invariant: row_ptr[lo] <= j < row_ptr[hi]
    while (hi - lo > 1) {
        const int32_t mid = (lo + hi) >> 1;
        if (row_ptr[mid] <= j) lo = mid; else hi = mid;
    }
    return lo;
}

__global__ void k_weights(const int64_t* __restrict__ row_ptr, int32_t vocab, int64_t nnz,
                          br_posting* __restrict__ post, const uint16_t* __restrict__ tf,
                          const uint32_t* __restrict__ dl, const double* __restrict__ idf, double avgdl,
                          double k1, double b, int variant, float* __restrict__ ub, float* __restrict__ amax) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    float wv = 0.f;
    const int32_t lo = warp_term_of(row_ptr, vocab, nnz, j, lane);
    if (lo >= 0) {
        const uint32_t d = post[j].doc;
        const double c = bm25_contrib(idf[lo], (double)tf[j], (double)dl[d], avgdl, k1, b, variant);
        wv = isnan(c) ? 0.f : (float)c;
        post[j].w = wv;
    }
    // ub[t] = max posting weight of term t (the score upper bound of the tiled scorer's deferral): one atomic per
    // (warp, term) - the lanes of a warp hold consecutive postings, i.e. mostly one term.  Weights < 0 (idf without
    // +1) count as 0; non-negative floats order like their bit patterns.  amax (when not null) gets max |w| the same way.
    unsigned todo = __ballot_sync(0xffffffffu, lo >= 0);
    while (todo) {
        const int leader = __ffs(todo) - 1;
        const int32_t t = __shfl_sync(0xffffffffu, lo, leader);
        const bool mine = lo == t;
        const unsigned mx = __reduce_max_sync(0xffffffffu, mine ? __float_as_uint(fmaxf(wv, 0.f)) : 0u);
        if (lane == leader) atomicMax(reinterpret_cast<unsigned*>(ub) + t, mx);
        if (amax) {
            const unsigned ma = __reduce_max_sync(0xffffffffu, mine ? __float_as_uint(fabsf(wv)) : 0u);
            if (lane == leader) atomicMax(reinterpret_cast<unsigned*>(amax) + t, ma);
        }
        todo &= ~__ballot_sync(0xffffffffu, mine);
    }
}

// Append: row_ptr and df of the grown index over the grown vocabulary.  Terms t >= the old vocabulary have no old
// postings; rp_old[v_old] = the old nnz.
__global__ void k_append_rows(const int64_t* __restrict__ rp_old, const uint32_t* __restrict__ df_old, int32_t v_old,
                              const int64_t* __restrict__ rp_new_part, const uint32_t* __restrict__ df_new_part,
                              int32_t vocab, int64_t* __restrict__ row_ptr, uint32_t* __restrict__ df) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > vocab) return;
    row_ptr[t] = rp_old[min(t, v_old)] + rp_new_part[t];
    if (t < vocab) df[t] = (t < v_old ? df_old[t] : 0u) + df_new_part[t];
}

// Append: posting j of the grown index.  Its term's row is the term's old postings followed by the new documents'
// postings (doc ids shifted by the old N), so every output posting has exactly one source posting: one 10-byte read and
// one 10-byte write per posting.  Weights are left 0 for br_index_finalize.
__global__ void k_append_merge(const int64_t* __restrict__ row_ptr, int32_t vocab, int64_t nnz,
                               const int64_t* __restrict__ rp_old, int32_t v_old, const br_posting* __restrict__ post_old,
                               const uint16_t* __restrict__ tf_old, const int64_t* __restrict__ rp_new_part,
                               const br_posting* __restrict__ post_new_part, const uint16_t* __restrict__ tf_new_part,
                               uint32_t n_docs_old, br_posting* __restrict__ post, uint16_t* __restrict__ tf) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int32_t t = warp_term_of(row_ptr, vocab, nnz, j, threadIdx.x & 31);
    if (t < 0) return;
    const int64_t off = j - row_ptr[t];
    const int64_t old_lo = rp_old[min(t, v_old)], old_len = t < v_old ? rp_old[t + 1] - old_lo : 0;
    br_posting p;
    uint16_t f;
    if (off < old_len) {
        p.doc = post_old[old_lo + off].doc;
        f = tf_old[old_lo + off];
    } else {
        const int64_t s = rp_new_part[t] + (off - old_len);
        p.doc = post_new_part[s].doc + n_docs_old;
        f = tf_new_part[s];
    }
    p.w = 0.f;
    post[j] = p;
    tf[j] = f;
}

// Remove.  Both compactions use tiles of RLE_TILE items (RLE_T threads x RLE_I); new_id[doc] == kRemovedDoc marks a removed
// doc.
constexpr uint32_t kRemovedDoc = 0xffffffffu;

__global__ void __launch_bounds__(RLE_T) k_docmap_count(const uint8_t* __restrict__ remove, const uint32_t* __restrict__ dl,
                                                        int64_t n, uint32_t* __restrict__ block_counts,
                                                        unsigned long long* __restrict__ sum_dl) {
    const int64_t base = (int64_t)blockIdx.x * RLE_TILE;
    uint32_t c = 0;
    unsigned long long s = 0;
#pragma unroll
    for (int j = 0; j < RLE_I; ++j) {
        const int64_t i = base + j * RLE_T + threadIdx.x;   // striped: coalesced, order irrelevant
        if (i < n && !remove[i]) {
            ++c;
            s += dl[i];
        }
    }
    uint32_t total;
    block_excl_scan(c, &total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(sum_dl, s);
}

__global__ void __launch_bounds__(RLE_T) k_docmap_emit(const uint8_t* __restrict__ remove, const uint32_t* __restrict__ dl,
                                                       int64_t n, const int64_t* __restrict__ block_off,
                                                       uint32_t* __restrict__ new_id, uint32_t* __restrict__ dl_new) {
    const int64_t base = (int64_t)blockIdx.x * RLE_TILE + (int64_t)threadIdx.x * RLE_I;  // blocked: ordered
    bool keep[RLE_I];
    uint32_t c = 0;
#pragma unroll
    for (int j = 0; j < RLE_I; ++j) {
        keep[j] = base + j < n && !remove[base + j];
        c += keep[j] ? 1u : 0u;
    }
    uint32_t total;
    uint32_t o = (uint32_t)block_off[blockIdx.x] + block_excl_scan(c, &total);   // new ids are < 2^31
#pragma unroll
    for (int j = 0; j < RLE_I; ++j) {
        if (base + j >= n) break;
        if (keep[j]) {
            new_id[base + j] = o;
            dl_new[o] = dl[base + j];
            ++o;
        } else {
            new_id[base + j] = kRemovedDoc;
        }
    }
}

// Posting tile layout: warp w reads postings [32 * RLE_I * w, 32 * RLE_I * (w + 1)) of the tile in RLE_I coalesced rounds of
// 32; round r of warp w is chunk w * RLE_I + r of the tile.
__global__ void __launch_bounds__(RLE_T) k_remove_count(const br_posting* __restrict__ post, int64_t nnz,
                                                        const uint32_t* __restrict__ new_id,
                                                        uint32_t* __restrict__ block_counts) {
    const int64_t base = (int64_t)blockIdx.x * RLE_TILE + (threadIdx.x >> 5) * (32 * RLE_I) + (threadIdx.x & 31);
    uint32_t c = 0;
#pragma unroll
    for (int r = 0; r < RLE_I; ++r) {
        const int64_t i = base + r * 32;
        if (i < nnz && new_id[post[i].doc] != kRemovedDoc) ++c;
    }
    uint32_t total;
    block_excl_scan(c, &total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// Writes the tile's surviving postings from block_off[tile] on, in order, with their new doc ids and weight 0 (for
// br_index_finalize), and row_ptr_new[t] = the number of survivors before row_ptr[t] for every term whose row starts in
// the tile; the last tile also takes the terms whose rows start at nnz (trailing empty rows and t = vocab).  The count
// before a position p of the tile is the prefix of its chunk plus a popcount of the chunk's keep ballot below p.
__global__ void __launch_bounds__(RLE_T) k_remove_emit(const int64_t* __restrict__ row_ptr, int32_t vocab,
                                                       const br_posting* __restrict__ post, const uint16_t* __restrict__ tf,
                                                       int64_t nnz, const uint32_t* __restrict__ new_id,
                                                       const int64_t* __restrict__ block_off,
                                                       br_posting* __restrict__ post_new, uint16_t* __restrict__ tf_new,
                                                       int64_t* __restrict__ row_ptr_new) {
    constexpr int NC = RLE_TILE / 32;                      // chunks of 32 postings per tile
    __shared__ uint32_t s_ballot[NC + 1], s_pre[NC + 1];   // [NC]: position RLE_TILE (the end of a full last tile)
    __shared__ int32_t s_terms[2];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t tile_lo = (int64_t)blockIdx.x * RLE_TILE;
    if (w == (RLE_T >> 5) - 1 && lane < 2) {
        // the terms whose rows start in the tile: [first t with row_ptr[t] >= tile_lo, first t with row_ptr[t] >= key)
        const int64_t key = lane == 0 ? tile_lo : (tile_lo + RLE_TILE >= nnz ? nnz + 1 : tile_lo + RLE_TILE);
        int32_t a = 0, b = vocab + 1;
        while (a < b) {
            const int32_t mid = (a + b) >> 1;
            if (row_ptr[mid] < key) a = mid + 1; else b = mid;
        }
        s_terms[lane] = a;
    }
    const int64_t base = tile_lo + w * (32 * RLE_I) + lane;
    uint32_t nid[RLE_I], bal[RLE_I];
    uint16_t f[RLE_I];
#pragma unroll
    for (int r = 0; r < RLE_I; ++r) {
        const int64_t i = base + r * 32;
        nid[r] = kRemovedDoc;
        f[r] = 0;
        if (i < nnz) {
            nid[r] = new_id[post[i].doc];
            f[r] = tf[i];
        }
        bal[r] = __ballot_sync(0xffffffffu, nid[r] != kRemovedDoc);
    }
    if (lane < RLE_I) {
        uint32_t mine = bal[0];
#pragma unroll
        for (int r = 1; r < RLE_I; ++r) if (lane == r) mine = bal[r];
        s_ballot[w * RLE_I + lane] = mine;
    }
    if (threadIdx.x == 0) s_ballot[NC] = 0;
    __syncthreads();
    if (w == 0) {                                          // exclusive prefix over the NC chunks, two per lane
        static_assert(NC == 64, "two chunks per lane of one warp");
        const uint32_t v0 = __popc(s_ballot[2 * lane]), v1 = __popc(s_ballot[2 * lane + 1]);
        const uint32_t incl = warp_incl_scan(v0 + v1, lane);
        s_pre[2 * lane] = incl - v0 - v1;
        s_pre[2 * lane + 1] = incl - v1;
        if (lane == 31) s_pre[NC] = incl;
    }
    __syncthreads();
    const int64_t out0 = block_off[blockIdx.x];
    const uint32_t below = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < RLE_I; ++r) {
        if (nid[r] != kRemovedDoc) {
            const int64_t o = out0 + s_pre[w * RLE_I + r] + __popc(bal[r] & below);
            br_posting p;
            p.doc = nid[r];
            p.w = 0.f;
            post_new[o] = p;
            tf_new[o] = f[r];
        }
    }
    for (int32_t t = s_terms[0] + threadIdx.x; t < s_terms[1]; t += RLE_T) {
        const uint32_t pos = (uint32_t)(row_ptr[t] - tile_lo);   // in [0, RLE_TILE]
        const uint32_t c = pos >> 5;
        row_ptr_new[t] = out0 + s_pre[c] + __popc(s_ballot[c] & ((1u << (pos & 31)) - 1u));
    }
}

__global__ void k_remove_df(const int64_t* __restrict__ row_ptr, int32_t vocab, uint32_t* __restrict__ df) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < vocab) df[t] = (uint32_t)(row_ptr[t + 1] - row_ptr[t]);
}

__global__ void k_skip(const int64_t* __restrict__ row_ptr, const br_posting* __restrict__ post,
                       const int32_t* __restrict__ hot_terms, int32_t n_hot, int32_t n_sub, int sub_shift,
                       uint32_t* __restrict__ skip) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t per = (int64_t)n_sub + 1;
    if (i >= (int64_t)n_hot * per) return;
    const int32_t slot = (int32_t)(i / per);
    const int64_t j = i - (int64_t)slot * per;
    const int32_t t = hot_terms[slot];
    const int64_t base = row_ptr[t];
    const uint32_t len = (uint32_t)(row_ptr[t + 1] - base);
    const uint64_t target = (uint64_t)j << sub_shift;   // first doc of sub-range j
    uint32_t lo = 0, hi = len;                           // first posting with doc >= target
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if ((uint64_t)post[base + mid].doc < target) lo = mid + 1; else hi = mid;
    }
    skip[i] = lo;
}

__global__ void k_rows_fill(const int64_t* __restrict__ row_ptr, const br_posting* __restrict__ post,
                            const int32_t* __restrict__ row_terms, int32_t n_rows, int64_t n_pad, float* __restrict__ rows) {
    const int r = blockIdx.y;
    if (r >= n_rows) return;
    const int32_t t = row_terms[r];
    const int64_t lo = row_ptr[t], n = row_ptr[t + 1] - lo;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const br_posting p = post[lo + i];
        rows[(int64_t)r * n_pad + p.doc] = p.w;
    }
}

// CSR validation for imported indexes (a truncated / corrupt file must not cause out-of-bounds accesses later):
// bit 1: row_ptr not monotone or outside [0, nnz]; bit 2: doc id outside [0, n_docs); bit 8: doc ids not strictly
// ascending inside a row; bit 4: tf == 0
__global__ void k_validate_rows(const int64_t* __restrict__ row_ptr, int32_t vocab, int64_t nnz, uint32_t* __restrict__ df,
                                int* __restrict__ bad) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= vocab) return;
    const int64_t a = row_ptr[t], b = row_ptr[t + 1];
    if (a < 0 || b < a || b > nnz || (t == 0 && a != 0) || (t == vocab - 1 && b != nnz)) { atomicOr(bad, 1); df[t] = 0; return; }
    df[t] = (uint32_t)(b - a);
}
__global__ void k_validate_postings(const int64_t* __restrict__ row_ptr, int32_t vocab, const int32_t* __restrict__ doc,
                                    const uint16_t* __restrict__ tf_in, int64_t nnz, int64_t n_docs,
                                    br_posting* __restrict__ post, uint16_t* __restrict__ tf, int* __restrict__ bad) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    const int32_t d = doc[j];
    if (d < 0 || d >= n_docs) atomicOr(bad, 2);
    if (tf_in[j] == 0) atomicOr(bad, 4);
    if (j > 0 && d <= doc[j - 1]) {
        // allowed only at the first posting of a row: is j some row_ptr[t]?
        int32_t lo = 0, hi = vocab;                       // last t with row_ptr[t] <= j
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (row_ptr[mid] <= j) lo = mid; else hi = mid;
        }
        if (row_ptr[lo] != j) atomicOr(bad, 8);
    }
    post[j].doc = (uint32_t)d;
    post[j].w = 0.f;
    tf[j] = tf_in[j];
}
__global__ void k_sum_dl(const int32_t* __restrict__ dl_in, int64_t n, uint32_t* __restrict__ dl, unsigned long long* __restrict__ sum,
                         int* __restrict__ bad) {
    unsigned long long s = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int32_t v = dl_in[i];
        if (v < 0) atomicOr(bad, 16);
        dl[i] = (uint32_t)v;
        s += (unsigned long long)max(v, 0);
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(sum, s);
}
__global__ void k_tf_to_u16(const int32_t* __restrict__ tf_in, int64_t nnz, uint16_t* __restrict__ out, int* __restrict__ bad) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    if (tf_in[j] < 0 || tf_in[j] > 65535) atomicOr(bad, 32);
    out[j] = (uint16_t)tf_in[j];
}
__global__ void k_export_u16(const br_posting* __restrict__ post, int64_t nnz, int32_t* __restrict__ doc_out) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < nnz) doc_out[j] = (int32_t)post[j].doc;
}

__global__ void k_export(const br_posting* __restrict__ post, const uint16_t* __restrict__ tf, int64_t nnz,
                         int32_t* __restrict__ doc_out, int32_t* __restrict__ tf_out) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nnz) return;
    doc_out[j] = (int32_t)post[j].doc;
    tf_out[j] = (int32_t)tf[j];
}

// ------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------


void index_free(br_index* ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);   // the members free their memory on the handle's device
    delete ix;
}

static int alloc_common(br_index* ix) {
    BR_TRY(ix->row_ptr.alloc((size_t)ix->vocab + 1));
    BR_TRY(ix->dl.alloc((size_t)ix->n_docs));
    BR_TRY(ix->df.alloc((size_t)ix->vocab));
    BR_TRY(ix->idf.alloc((size_t)ix->vocab));
    BR_TRY(ix->hot_slot.alloc((size_t)ix->vocab));
    BR_TRY(ix->ub.alloc((size_t)ix->vocab));
    return BR_OK;
}

using IndexOwner = std::unique_ptr<br_index, decltype(&index_free)>;   // a half-built handle: freed unless released

int index_build(const int32_t* tok, const int64_t* doc_off, int64_t n_docs, int32_t vocab, int64_t doc_base,
                cudaStream_t st, br_index** out) {
    BR_REQUIRE(out && tok && doc_off, BR_ERR_INVALID, "br_index_build: null pointer");
    BR_REQUIRE(n_docs > 0 && n_docs < (1LL << 31), BR_ERR_INVALID,
               "br_index_build: n_docs must be in [1, 2^31) (empty corpus: the reference divides by zero, "
               "bm25_ranking.ipynb:171)");
    BR_REQUIRE(vocab > 0, BR_ERR_INVALID, "br_index_build: vocab must be positive");
    *out = nullptr;
    IndexOwner ix(new br_index(), index_free);
    BR_CUDA(cudaGetDevice(&ix->device));
    ix->n_docs = n_docs; ix->vocab = vocab; ix->doc_base = doc_base;

    int64_t n_tok = 0;
    BR_CUDA(cudaMemcpyAsync(&n_tok, doc_off + n_docs, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(n_tok >= 0 && n_tok < (1LL << 32), BR_ERR_UNSUPPORTED,
               "br_index_build: more than 2^32 tokens in one shard");
    ix->sum_dl = n_tok;
    BR_TRY(alloc_common(ix.get()));

    DevArray<int> d_bad;
    DevArray<uint32_t> keys_a, keys_b, vals_a, vals_b, block_counts, post_term, head_pos, tstart, tend;
    DevArray<int64_t> block_off;
    DevArray<unsigned char> sort_tmp;
    BR_TRY(d_bad.alloc(1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    BR_TRY(keys_a.alloc((size_t)n_tok));
    BR_TRY(keys_b.alloc((size_t)n_tok));
    BR_TRY(vals_a.alloc((size_t)n_tok));
    BR_TRY(vals_b.alloc((size_t)n_tok));
    k_make_keys<<<kNumSMs * 8, 256, 0, st>>>(tok, doc_off, n_docs, vocab, keys_a, vals_a, ix->dl, d_bad);
    BR_CUDA(cudaGetLastError());

    // STABLE sort of (term, doc) pairs by the significant bits of the term alone: the tokens arrive in doc order, so
    // inside a term the docs stay ascending and the occurrences of one (term, doc) stay adjacent - 3 radix passes for a
    // 1M-term vocabulary instead of 7 over a 52-bit (term, doc) key
    int term_bits = 1;
    while ((1LL << term_bits) < (int64_t)vocab) ++term_bits;
    cub::DoubleBuffer<uint32_t> dkeys(keys_a, keys_b), dvals(vals_a, vals_b);
    size_t tmp_bytes = 0;
    BR_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, dkeys, dvals, (int64_t)n_tok, 0, term_bits, st));
    BR_TRY(sort_tmp.alloc(tmp_bytes + 16));
    BR_CUDA(cub::DeviceRadixSort::SortPairs(sort_tmp, tmp_bytes, dkeys, dvals, (int64_t)n_tok, 0, term_bits, st));
    const uint32_t* keys = dkeys.Current();
    const uint32_t* vals = dvals.Current();

    // run-length encode
    const int64_t n_blocks = (n_tok + RLE_TILE - 1) / RLE_TILE;
    BR_TRY(block_counts.alloc((size_t)n_blocks + 1));
    BR_TRY(block_off.alloc((size_t)n_blocks + 2));
    if (n_blocks > 0) {
        k_rle_count<<<(unsigned)n_blocks, RLE_T, 0, st>>>(keys, vals, n_tok, block_counts);
        BR_CUDA(cudaGetLastError());
    }
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(block_counts, n_blocks, block_off);
    BR_CUDA(cudaGetLastError());
    int64_t nnz = 0;
    int bad = 0;
    BR_CUDA(cudaMemcpyAsync(&nnz, block_off + n_blocks, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!(bad & 1), BR_ERR_INVALID, "br_index_build: token id outside [0, vocab)");
    BR_REQUIRE(!(bad & 2), BR_ERR_INVALID, "br_index_build: doc_offsets not non-decreasing");
    ix->nnz = nnz;
    BR_TRY(ix->post.alloc((size_t)nnz));
    BR_TRY(ix->tf.alloc((size_t)nnz));
    BR_TRY(post_term.alloc((size_t)nnz));
    BR_TRY(head_pos.alloc((size_t)nnz));
    BR_TRY(tstart.alloc((size_t)vocab));
    BR_TRY(tend.alloc((size_t)vocab));
    BR_CUDA(cudaMemsetAsync(tstart, 0, sizeof(uint32_t) * (size_t)vocab, st));
    BR_CUDA(cudaMemsetAsync(tend, 0, sizeof(uint32_t) * (size_t)vocab, st));
    if (n_blocks > 0) {
        k_rle_emit<<<(unsigned)n_blocks, RLE_T, 0, st>>>(keys, vals, n_tok, block_off, ix->post, post_term, head_pos);
        BR_CUDA(cudaGetLastError());
    }
    if (nnz > 0) {
        k_finish<<<blocks_for(nnz, 256), 256, 0, st>>>(post_term, head_pos, nnz, (uint32_t)n_tok, ix->tf, tstart,
                                                       tend, d_bad);
        BR_CUDA(cudaGetLastError());
    }
    k_df<<<blocks_for(vocab, 256), 256, 0, st>>>(tstart, tend, vocab, ix->df);
    BR_CUDA(cudaGetLastError());
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(ix->df, vocab, ix->row_ptr);
    BR_CUDA(cudaGetLastError());
    ix->h_df.resize((size_t)vocab);
    BR_CUDA(cudaMemcpyAsync(ix->h_df.data(), ix->df, sizeof(uint32_t) * (size_t)vocab, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!(bad & 4), BR_ERR_UNSUPPORTED, "br_index_build: a term occurs more than 65535 times in one doc");
    *out = ix.release();
    return BR_OK;
}

// Import from DEVICE arrays (the flat index file is staged through pinned memory by the caller): validates the CSR on the
// device, copies it into library-owned arrays.  Call index_finalize afterwards.
int index_import_dev(const int64_t* row_ptr, const int32_t* doc, const uint16_t* tf, const int32_t* dl, int64_t n_docs,
                     int32_t vocab, int64_t nnz, int64_t doc_base, cudaStream_t st, br_index** out) {
    BR_REQUIRE(out && row_ptr && dl && (nnz == 0 || (doc && tf)), BR_ERR_INVALID, "br_index_import_csr_dev: null pointer");
    BR_REQUIRE(n_docs > 0 && n_docs < (1LL << 31) && vocab > 0 && nnz >= 0 && nnz < (1LL << 32), BR_ERR_INVALID,
               "br_index_import_csr_dev: bad sizes");
    *out = nullptr;
    IndexOwner ix(new br_index(), index_free);
    BR_CUDA(cudaGetDevice(&ix->device));
    ix->n_docs = n_docs; ix->vocab = vocab; ix->doc_base = doc_base; ix->nnz = nnz;
    BR_TRY(alloc_common(ix.get()));
    BR_TRY(ix->post.alloc((size_t)nnz));
    BR_TRY(ix->tf.alloc((size_t)nnz));
    DevArray<int> d_bad;
    DevArray<unsigned long long> d_sum;
    BR_TRY(d_bad.alloc(1));
    BR_TRY(d_sum.alloc(1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    BR_CUDA(cudaMemsetAsync(d_sum, 0, sizeof(unsigned long long), st));
    BR_CUDA(cudaMemcpyAsync(ix->row_ptr, row_ptr, sizeof(int64_t) * ((size_t)vocab + 1), cudaMemcpyDeviceToDevice, st));
    k_validate_rows<<<blocks_for(vocab, 256), 256, 0, st>>>(ix->row_ptr, vocab, nnz, ix->df, d_bad);
    BR_CUDA(cudaGetLastError());
    int bad = 0;
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));                  // row_ptr must be sound before the posting pass searches it
    BR_REQUIRE(!bad, BR_ERR_INVALID, "br_index_import_csr: row_ptr is not a monotone [0 .. nnz] offset array");
    if (nnz > 0) {
        k_validate_postings<<<blocks_for(nnz, 256), 256, 0, st>>>(ix->row_ptr, vocab, doc, tf, nnz, n_docs, ix->post, ix->tf, d_bad);
        BR_CUDA(cudaGetLastError());
    }
    k_sum_dl<<<kNumSMs * 4, 256, 0, st>>>(dl, n_docs, ix->dl, d_sum, d_bad);
    BR_CUDA(cudaGetLastError());
    ix->h_df.resize((size_t)vocab);
    unsigned long long sum = 0;
    BR_CUDA(cudaMemcpyAsync(ix->h_df.data(), ix->df, sizeof(uint32_t) * (size_t)vocab, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&sum, d_sum, sizeof(sum), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!(bad & 2), BR_ERR_INVALID, "br_index_import_csr: doc id outside [0, n_docs)");
    BR_REQUIRE(!(bad & 8), BR_ERR_INVALID, "br_index_import_csr: doc ids not strictly ascending inside a posting list");
    BR_REQUIRE(!(bad & 4), BR_ERR_INVALID, "br_index_import_csr: tf outside [1, 65535]");
    BR_REQUIRE(!(bad & 16), BR_ERR_INVALID, "br_index_import_csr: negative doc length");
    ix->sum_dl = (int64_t)sum;
    *out = ix.release();
    return BR_OK;
}

// Import from HOST arrays (unpickling): upload, then the same validation.
int index_import(const int64_t* row_ptr, const int32_t* doc, const int32_t* tf, const int32_t* dl, int64_t n_docs,
                 int32_t vocab, int64_t doc_base, cudaStream_t st, br_index** out) {
    BR_REQUIRE(out && row_ptr && doc && tf && dl, BR_ERR_INVALID, "br_index_import_csr: null pointer");
    BR_REQUIRE(n_docs > 0 && n_docs < (1LL << 31) && vocab > 0, BR_ERR_INVALID, "br_index_import_csr: bad sizes");
    *out = nullptr;
    const int64_t nnz = row_ptr[vocab];
    BR_REQUIRE(nnz >= 0 && nnz < (1LL << 32) && row_ptr[0] == 0, BR_ERR_INVALID, "br_index_import_csr: bad row_ptr");
    DevArray<int64_t> d_rp;
    DevArray<int32_t> d_doc, d_tf, d_dl;
    DevArray<uint16_t> d_tf16;
    DevArray<int> d_bad;
    BR_TRY(d_rp.alloc((size_t)vocab + 1));
    BR_TRY(d_doc.alloc((size_t)nnz));
    BR_TRY(d_tf.alloc((size_t)nnz));
    BR_TRY(d_tf16.alloc((size_t)nnz));
    BR_TRY(d_dl.alloc((size_t)n_docs));
    BR_TRY(d_bad.alloc(1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    BR_CUDA(cudaMemcpyAsync(d_rp, row_ptr, sizeof(int64_t) * ((size_t)vocab + 1), cudaMemcpyHostToDevice, st));
    BR_CUDA(cudaMemcpyAsync(d_doc, doc, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    BR_CUDA(cudaMemcpyAsync(d_tf, tf, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    BR_CUDA(cudaMemcpyAsync(d_dl, dl, sizeof(int32_t) * (size_t)n_docs, cudaMemcpyHostToDevice, st));
    if (nnz > 0) {
        k_tf_to_u16<<<blocks_for(nnz, 256), 256, 0, st>>>(d_tf, nnz, d_tf16, d_bad);
        BR_CUDA(cudaGetLastError());
    }
    int bad = 0;
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!bad, BR_ERR_INVALID, "br_index_import_csr: tf outside [0, 65535]");
    return index_import_dev(d_rp, d_doc, d_tf16, d_dl, n_docs, vocab, nnz, doc_base, st, out);
}

// Append documents: the new documents' postings come from index_build (the same sort and run-length encoding, over the
// grown vocabulary), then one streaming pass merges them behind each term's old postings.  Every grown array is
// allocated and filled before any of them replaces the handle's, so that an error leaves the handle as it was.
int index_append(br_index* ix, const int32_t* tok, const int64_t* doc_off, int64_t n_docs, int32_t vocab,
                 cudaStream_t st) {
    BR_REQUIRE(ix && tok && doc_off, BR_ERR_INVALID, "br_index_append: null pointer");
    BR_REQUIRE(n_docs > 0 && n_docs < (1LL << 31), BR_ERR_INVALID, "br_index_append: n_docs must be in [1, 2^31)");
    BR_REQUIRE(vocab >= ix->vocab, BR_ERR_INVALID, "br_index_append: vocab must be at least the index's vocab");
    BR_CUDA(cudaSetDevice(ix->device));
    br_index* part_raw = nullptr;
    BR_TRY(index_build(tok, doc_off, n_docs, vocab, 0, st, &part_raw));
    IndexOwner part(part_raw, index_free);
    const int64_t n_docs_new = ix->n_docs + n_docs, sum_dl = ix->sum_dl + part->sum_dl, nnz = ix->nnz + part->nnz;
    BR_REQUIRE(n_docs_new < (1LL << 31), BR_ERR_UNSUPPORTED, "br_index_append: 2^31 or more docs in one shard");
    BR_REQUIRE(sum_dl < (1LL << 32), BR_ERR_UNSUPPORTED, "br_index_append: 2^32 or more tokens in one shard");
    BR_REQUIRE(nnz < (1LL << 32), BR_ERR_UNSUPPORTED, "br_index_append: 2^32 or more postings in one shard");

    const size_t V = (size_t)vocab;
    const bool grow_v = vocab > ix->vocab;
    DevArray<int64_t> row_ptr;
    DevArray<br_posting> post;
    DevArray<uint16_t> tf;
    DevArray<uint32_t> dl, df;
    DevArray<double> idf;
    DevArray<int32_t> hot_slot;
    DevArray<float> ub;
    BR_TRY(row_ptr.alloc(V + 1));
    BR_TRY(df.alloc(V));
    BR_TRY(dl.alloc((size_t)n_docs_new));
    BR_TRY(post.alloc((size_t)nnz));
    BR_TRY(tf.alloc((size_t)nnz));
    if (grow_v) {
        BR_TRY(idf.alloc(V));
        BR_TRY(hot_slot.alloc(V));
        BR_TRY(ub.alloc(V));
    }
    k_append_rows<<<blocks_for((int64_t)V + 1, 256), 256, 0, st>>>(ix->row_ptr, ix->df, ix->vocab, part->row_ptr, part->df,
                                                                   vocab, row_ptr, df);
    BR_CUDA(cudaGetLastError());
    if (nnz > 0) {
        k_append_merge<<<blocks_for(nnz, 256), 256, 0, st>>>(row_ptr, vocab, nnz, ix->row_ptr, ix->vocab, ix->post, ix->tf,
                                                             part->row_ptr, part->post, part->tf, (uint32_t)ix->n_docs,
                                                             post, tf);
        BR_CUDA(cudaGetLastError());
    }
    BR_CUDA(cudaMemcpyAsync(dl, ix->dl, sizeof(uint32_t) * (size_t)ix->n_docs, cudaMemcpyDeviceToDevice, st));
    BR_CUDA(cudaMemcpyAsync(dl + ix->n_docs, part->dl, sizeof(uint32_t) * (size_t)n_docs, cudaMemcpyDeviceToDevice, st));
    std::vector<uint32_t> h_df(V);
    BR_CUDA(cudaMemcpyAsync(h_df.data(), df, sizeof(uint32_t) * V, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));

    // nothing below can fail: the handle takes the grown arrays and frees the old ones
    ix->row_ptr = std::move(row_ptr);
    ix->post = std::move(post);
    ix->tf = std::move(tf);
    ix->dl = std::move(dl);
    ix->df = std::move(df);
    ix->h_df.swap(h_df);
    if (grow_v) {
        ix->idf = std::move(idf);
        ix->hot_slot = std::move(hot_slot);
        ix->ub = std::move(ub);
        ix->amax.reset();       // [V] arrays that index_finalize allocates when they are missing
        ix->row_slot.reset();
    }
    // structures index_finalize builds only when they are missing: they depend on the local df and N
    ix->skip.reset();
    ix->sig_bit.reset();
    ix->dense_rows.reset();
    ix->n_rows = ix->n_srows = 0;
    ix->post_cos.reset();
    ix->cos_inv_norm.reset();
    ix->n_docs = n_docs_new;
    ix->vocab = vocab;
    ix->sum_dl = sum_dl;
    ix->nnz = nnz;
    ix->finalized = false;
    return BR_OK;
}

// Remove documents: compact the docs (new id = rank among the kept docs), then the postings, which keeps every row's docs
// ascending.  Terms keep their ids; a term that loses all its postings keeps an empty row.  As in index_append, every
// new array is allocated and filled before any of them replaces the handle's, so that an error leaves the handle as it
// was.
int index_remove(br_index* ix, const uint8_t* remove, cudaStream_t st) {
    BR_REQUIRE(ix && remove, BR_ERR_INVALID, "br_index_remove: null pointer");
    BR_CUDA(cudaSetDevice(ix->device));
    const int64_t N = ix->n_docs, nnz = ix->nnz;
    const size_t V = (size_t)ix->vocab;

    // doc map
    const int64_t nb_docs = (N + RLE_TILE - 1) / RLE_TILE;
    DevArray<uint32_t> new_id, doc_counts, post_counts, dl, df;
    DevArray<int64_t> doc_off, post_off, row_ptr;
    DevArray<unsigned long long> d_sum;
    BR_TRY(new_id.alloc((size_t)N));
    BR_TRY(doc_counts.alloc((size_t)nb_docs));
    BR_TRY(doc_off.alloc((size_t)nb_docs + 1));
    BR_TRY(d_sum.alloc(1));
    BR_CUDA(cudaMemsetAsync(d_sum, 0, sizeof(unsigned long long), st));
    k_docmap_count<<<(unsigned)nb_docs, RLE_T, 0, st>>>(remove, ix->dl, N, doc_counts, d_sum);
    BR_CUDA(cudaGetLastError());
    k_exscan<uint32_t><<<1, 1024, 0, st>>>(doc_counts, nb_docs, doc_off);
    BR_CUDA(cudaGetLastError());
    int64_t n_kept = 0;
    unsigned long long sum_dl = 0;
    BR_CUDA(cudaMemcpyAsync(&n_kept, doc_off + nb_docs, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&sum_dl, d_sum, sizeof(sum_dl), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    if (n_kept == N) return BR_OK;                         // nothing to remove: the handle stays as it is, finalised
    BR_REQUIRE(n_kept > 0, BR_ERR_INVALID, "br_index_remove: every document would be removed (an index holds at least one)");
    BR_TRY(dl.alloc((size_t)n_kept));
    k_docmap_emit<<<(unsigned)nb_docs, RLE_T, 0, st>>>(remove, ix->dl, N, doc_off, new_id, dl);
    BR_CUDA(cudaGetLastError());

    // postings
    const int64_t nb_post = (nnz + RLE_TILE - 1) / RLE_TILE;
    int64_t nnz_new = 0;
    BR_TRY(row_ptr.alloc(V + 1));
    BR_TRY(df.alloc(V));
    BR_TRY(post_counts.alloc((size_t)nb_post));
    BR_TRY(post_off.alloc((size_t)nb_post + 1));
    if (nnz > 0) {
        k_remove_count<<<(unsigned)nb_post, RLE_T, 0, st>>>(ix->post, nnz, new_id, post_counts);
        BR_CUDA(cudaGetLastError());
        k_exscan<uint32_t><<<1, 1024, 0, st>>>(post_counts, nb_post, post_off);
        BR_CUDA(cudaGetLastError());
        BR_CUDA(cudaMemcpyAsync(&nnz_new, post_off + nb_post, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        BR_CUDA(cudaStreamSynchronize(st));
    }
    DevArray<br_posting> post;
    DevArray<uint16_t> tf;
    BR_TRY(post.alloc((size_t)nnz_new));
    BR_TRY(tf.alloc((size_t)nnz_new));
    if (nnz > 0) {
        k_remove_emit<<<(unsigned)nb_post, RLE_T, 0, st>>>(ix->row_ptr, ix->vocab, ix->post, ix->tf, nnz, new_id, post_off,
                                                            post, tf, row_ptr);
        BR_CUDA(cudaGetLastError());
    } else {
        BR_CUDA(cudaMemsetAsync(row_ptr, 0, sizeof(int64_t) * (V + 1), st));
    }
    k_remove_df<<<blocks_for((int64_t)V, 256), 256, 0, st>>>(row_ptr, ix->vocab, df);
    BR_CUDA(cudaGetLastError());
    std::vector<uint32_t> h_df(V);
    BR_CUDA(cudaMemcpyAsync(h_df.data(), df, sizeof(uint32_t) * V, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));

    // nothing below can fail: the handle takes the compacted arrays and frees the old ones
    ix->row_ptr = std::move(row_ptr);
    ix->post = std::move(post);
    ix->tf = std::move(tf);
    ix->dl = std::move(dl);
    ix->df = std::move(df);
    ix->h_df.swap(h_df);
    // structures index_finalize builds only when they are missing: they depend on the local df and N
    ix->skip.reset();
    ix->sig_bit.reset();
    ix->dense_rows.reset();
    ix->n_rows = ix->n_srows = 0;
    ix->post_cos.reset();
    ix->cos_inv_norm.reset();
    ix->n_docs = n_kept;
    ix->sum_dl = (int64_t)sum_dl;
    ix->nnz = nnz_new;
    ix->finalized = false;
    return BR_OK;
}

int index_finalize(br_index* ix, double k1, double b, int variant, double n_stat, double sum_dl_stat,
                   const int64_t* df_stat_host, cudaStream_t st) {
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_index_finalize: null handle");
    BR_REQUIRE(variant >= 0 && variant <= 2, BR_ERR_INVALID, "br_index_finalize: unknown variant");
    BR_CUDA(cudaSetDevice(ix->device));
    ix->post_cos.reset();                    // the TF-IDF tables depend on idf: rebuilt on demand after a re-finalise
    ix->cos_inv_norm.reset();
    ix->k1 = k1; ix->b = b; ix->variant = variant;
    ix->n_stat = n_stat > 0 ? n_stat : (double)ix->n_docs;
    const double sum_dl = sum_dl_stat > 0 ? sum_dl_stat : (double)ix->sum_dl;
    ix->sum_dl_stat = sum_dl;
    ix->avgdl = sum_dl / ix->n_stat;                       // sum(len(doc)) / corpus_size, :171
    const size_t V = (size_t)ix->vocab;
    ix->h_df_stat.resize(V);
    ix->h_idf.resize(V);
    {   // idf on the host: libm log() is the routine behind math.log (:189) - bit-identical, unlike the device's log();
        // V evaluations split over a few threads
        const unsigned nth = (unsigned)std::max<size_t>(1, std::min<size_t>({(size_t)16, (size_t)std::thread::hardware_concurrency(), V / 65536 + 1}));
        auto work = [&](size_t lo, size_t hi) {
            for (size_t t = lo; t < hi; ++t) {
                const int64_t d = df_stat_host ? df_stat_host[t] : (int64_t)ix->h_df[t];
                ix->h_df_stat[t] = d;
                if (d > 0) {
                    const double x = (ix->n_stat - (double)d + 0.5) / ((double)d + 0.5);
                    ix->h_idf[t] = variant == BR_OKAPI_NO_PLUS1 ? log(x) : log(1 + x);
                } else {
                    ix->h_idf[t] = NAN;
                }
            }
        };
        std::vector<std::thread> th;
        const size_t per = (V + nth - 1) / nth;
        for (unsigned i = 1; i < nth; ++i) th.emplace_back(work, std::min(V, i * per), std::min(V, (i + 1) * per));
        work(0, std::min(V, per));
        for (auto& x : th) x.join();
    }
    BR_CUDA(cudaMemcpyAsync(ix->idf, ix->h_idf.data(), sizeof(double) * V, cudaMemcpyHostToDevice, st));
    BR_CUDA(cudaMemsetAsync(ix->ub, 0, sizeof(float) * V, st));
    // only okapi_no_plus1 has negative idf, i.e. queries whose weights can have mixed signs (br_query.cu)
    if (variant == BR_OKAPI_NO_PLUS1) {
        if (!ix->amax) BR_TRY(ix->amax.alloc(V));
        BR_CUDA(cudaMemsetAsync(ix->amax, 0, sizeof(float) * V, st));
    } else {
        ix->amax.reset();
    }
    if (ix->nnz > 0) {
        k_weights<<<blocks_for(ix->nnz, 256), 256, 0, st>>>(ix->row_ptr, ix->vocab, ix->nnz, ix->post, ix->tf,
                                                            ix->dl, ix->idf, ix->avgdl, k1, b, variant, ix->ub, ix->amax);
        BR_CUDA(cudaGetLastError());
    }
    // hot-term skip tables (shard-local structure: decided from the local df)
    if (!ix->skip) {
        ix->sub_shift = kSubShift;                       // docs per sub-range (= TILE_SHIFT of br_tile.cu)
        ix->n_sub = (int32_t)((ix->n_docs + (1LL << ix->sub_shift) - 1) >> ix->sub_shift);
        const uint32_t hot_min = (uint32_t)fmax(4.0, 0.25 * (double)ix->n_sub);
        ix->hot_min = hot_min;
        std::vector<int32_t> slot(V, -1), hot_terms;
        for (size_t t = 0; t < V; ++t)
            if (ix->h_df[t] >= hot_min) { slot[t] = (int32_t)hot_terms.size(); hot_terms.push_back((int32_t)t); }
        ix->n_hot = (int32_t)hot_terms.size();
        BR_CUDA(cudaMemcpyAsync(ix->hot_slot, slot.data(), sizeof(int32_t) * V, cudaMemcpyHostToDevice, st));
        if (ix->n_hot > 0) {
            const int64_t n_entries = (int64_t)ix->n_hot * ((int64_t)ix->n_sub + 1);
            DevArray<int32_t> d_hot;
            BR_TRY(ix->skip.alloc((size_t)n_entries));
            BR_TRY(d_hot.alloc((size_t)ix->n_hot));
            BR_CUDA(cudaMemcpyAsync(d_hot, hot_terms.data(), sizeof(int32_t) * (size_t)ix->n_hot,
                                    cudaMemcpyHostToDevice, st));
            k_skip<<<blocks_for(n_entries, 256), 256, 0, st>>>(ix->row_ptr, ix->post, d_hot, ix->n_hot, ix->n_sub,
                                                               ix->sub_shift, ix->skip);
            BR_CUDA(cudaGetLastError());
            BR_CUDA(cudaStreamSynchronize(st));
        }
    }
    {   // dense rows (rebuilt at every finalize: they hold the weights)
        double frac = 0.2;                       // streamed rows
        const double look_frac = 1.0 / 64.0;     // look-up rows
        std::vector<int32_t> cand_terms;
        for (size_t t = 0; t < V; ++t)
            if (ix->n_hot > 0 && (double)ix->h_df[t] >= look_frac * (double)ix->n_docs && ix->h_df[t] >= ix->hot_min)
                cand_terms.push_back((int32_t)t);
        std::sort(cand_terms.begin(), cand_terms.end(), [&](int32_t x, int32_t y) {
            return ix->h_df[(size_t)x] != ix->h_df[(size_t)y] ? ix->h_df[(size_t)x] > ix->h_df[(size_t)y] : x < y;
        });
        ix->n_pad = ((ix->n_docs + 4095) / 4096) * 4096;
        // at most 384 rows and 16 GiB (C4: ~260 rows x 35 MB = 9 GB of the 180 GB)
        const size_t max_rows = std::min<size_t>(384, (size_t)((16LL << 30) / (4 * ix->n_pad)));
        if (cand_terms.size() > max_rows) cand_terms.resize(max_rows);
        int32_t n_s = 0;
        for (int32_t t : cand_terms)
            if ((double)ix->h_df[(size_t)t] >= frac * (double)ix->n_docs && n_s < 32) ++n_s;
        ix->dense_rows.reset();
        ix->n_rows = (int32_t)cand_terms.size();
        ix->n_srows = n_s;
        std::vector<int16_t> slot(V, (int16_t)-1);
        for (size_t r = 0; r < cand_terms.size(); ++r) slot[(size_t)cand_terms[r]] = (int16_t)r;
        if (!ix->row_slot) BR_TRY(ix->row_slot.alloc(V));
        BR_CUDA(cudaMemcpyAsync(ix->row_slot, slot.data(), sizeof(int16_t) * V, cudaMemcpyHostToDevice, st));
        if (ix->n_rows > 0) {
            DevArray<int32_t> d_terms;
            BR_TRY(ix->dense_rows.alloc((size_t)ix->n_rows * (size_t)ix->n_pad));
            BR_TRY(d_terms.alloc((size_t)ix->n_rows));
            BR_CUDA(cudaMemsetAsync(ix->dense_rows, 0, sizeof(float) * (size_t)ix->n_rows * (size_t)ix->n_pad, st));
            BR_CUDA(cudaMemcpyAsync(d_terms, cand_terms.data(), sizeof(int32_t) * (size_t)ix->n_rows, cudaMemcpyHostToDevice, st));
            k_rows_fill<<<dim3(kNumSMs * 4, (unsigned)ix->n_rows), 256, 0, st>>>(ix->row_ptr, ix->post, d_terms, ix->n_rows, ix->n_pad,
                                                                              ix->dense_rows);
            BR_CUDA(cudaGetLastError());
            BR_CUDA(cudaStreamSynchronize(st));
        }
        BR_CUDA(cudaStreamSynchronize(st));
    }
    if (!ix->sig_bit) {
        // the 32 most frequent terms: the tiled scorer orders its queries by which of them they contain (br_tile.cu)
        std::vector<int32_t> order(V);
        for (size_t t = 0; t < V; ++t) order[t] = (int32_t)t;
        const size_t top = std::min<size_t>(32, V);
        std::partial_sort(order.begin(), order.begin() + top, order.end(), [&](int32_t x, int32_t y) {
            return ix->h_df[(size_t)x] != ix->h_df[(size_t)y] ? ix->h_df[(size_t)x] > ix->h_df[(size_t)y] : x < y;
        });
        std::vector<int8_t> bit(V, (int8_t)-1);
        for (size_t r = 0; r < top; ++r)
            if (ix->h_df[(size_t)order[r]] > 0) bit[(size_t)order[r]] = (int8_t)r;
        BR_TRY(ix->sig_bit.alloc(V));
        BR_CUDA(cudaMemcpyAsync(ix->sig_bit, bit.data(), V, cudaMemcpyHostToDevice, st));
        BR_CUDA(cudaStreamSynchronize(st));
    }
    BR_CUDA(cudaStreamSynchronize(st));
    ix->finalized = true;
    return BR_OK;
}

}  // namespace br

// ------------------------------------------------------------------------------------------
// C ABI (build / export side)
// ------------------------------------------------------------------------------------------
extern "C" {

int br_index_build(const int32_t* token_ids_dev, const int64_t* doc_offsets_dev, int64_t n_docs, int32_t vocab,
                   int64_t doc_base, void* stream, br_index** out) {
    return br::index_build(token_ids_dev, doc_offsets_dev, n_docs, vocab, doc_base, (cudaStream_t)stream, out);
}

int br_index_append(br_index* ix, const int32_t* token_ids_dev, const int64_t* doc_offsets_dev, int64_t n_docs,
                    int32_t vocab, void* stream) {
    return br::index_append(ix, token_ids_dev, doc_offsets_dev, n_docs, vocab, (cudaStream_t)stream);
}

int br_index_remove(br_index* ix, const uint8_t* remove_dev, void* stream) {
    return br::index_remove(ix, remove_dev, (cudaStream_t)stream);
}

int br_index_finalize(br_index* ix, double k1, double b, int variant, double n_stat, double sum_dl_stat,
                      const int64_t* df_stat_host, void* stream) {
    return br::index_finalize(ix, k1, b, variant, n_stat, sum_dl_stat, df_stat_host, (cudaStream_t)stream);
}

int br_index_import_csr(const int64_t* row_ptr_host, const int32_t* doc_host, const int32_t* tf_host,
                        const int32_t* dl_host, int64_t n_docs, int32_t vocab, int64_t doc_base, void* stream,
                        br_index** out) {
    return br::index_import(row_ptr_host, doc_host, tf_host, dl_host, n_docs, vocab, doc_base,
                            (cudaStream_t)stream, out);
}

int br_index_import_csr_dev(const int64_t* row_ptr_dev, const int32_t* doc_dev, const uint16_t* tf_dev, const int32_t* dl_dev,
                            int64_t n_docs, int32_t vocab, int64_t nnz, int64_t doc_base, void* stream, br_index** out) {
    return br::index_import_dev(row_ptr_dev, doc_dev, tf_dev, dl_dev, n_docs, vocab, nnz, doc_base, (cudaStream_t)stream, out);
}

int br_index_export_csr_dev(const br_index* ix, int64_t* row_ptr_dev, int32_t* doc_dev, uint16_t* tf_dev, int32_t* dl_dev,
                            void* stream) {
    BR_REQUIRE(ix && row_ptr_dev && dl_dev && (ix->nnz == 0 || (doc_dev && tf_dev)), BR_ERR_INVALID,
               "br_index_export_csr_dev: null pointer");
    BR_CUDA(cudaSetDevice(ix->device));
    cudaStream_t st = (cudaStream_t)stream;
    BR_CUDA(cudaMemcpyAsync(row_ptr_dev, ix->row_ptr, sizeof(int64_t) * ((size_t)ix->vocab + 1), cudaMemcpyDeviceToDevice, st));
    BR_CUDA(cudaMemcpyAsync(dl_dev, ix->dl, sizeof(uint32_t) * (size_t)ix->n_docs, cudaMemcpyDeviceToDevice, st));
    if (ix->nnz > 0) {
        BR_CUDA(cudaMemcpyAsync(tf_dev, ix->tf, sizeof(uint16_t) * (size_t)ix->nnz, cudaMemcpyDeviceToDevice, st));
        br::k_export_u16<<<br::blocks_for(ix->nnz, 256), 256, 0, st>>>(ix->post, ix->nnz, doc_dev);
        BR_CUDA(cudaGetLastError());
    }
    return BR_OK;
}

void br_index_destroy(br_index* ix) { br::index_free(ix); }

int br_index_stats(const br_index* ix, int64_t* n_docs, int32_t* vocab, int64_t* nnz, double* avgdl,
                   int64_t* sum_dl, int64_t* doc_base) {
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_index_stats: null handle");
    if (n_docs) *n_docs = ix->n_docs;
    if (vocab) *vocab = ix->vocab;
    if (nnz) *nnz = ix->nnz;
    if (avgdl) *avgdl = ix->finalized ? ix->avgdl : (double)ix->sum_dl / (double)ix->n_docs;
    if (sum_dl) *sum_dl = ix->sum_dl;
    if (doc_base) *doc_base = ix->doc_base;
    return BR_OK;
}

const uint32_t* br_index_df_dev(const br_index* ix) { return ix ? ix->df.get() : nullptr; }

int br_index_stats_in_force(const br_index* ix, double* n_stat, double* sum_dl_stat) {
    BR_REQUIRE(ix && ix->finalized, BR_ERR_STATE, "br_index_stats_in_force: call br_index_finalize first");
    if (n_stat) *n_stat = ix->n_stat;
    if (sum_dl_stat) *sum_dl_stat = ix->sum_dl_stat;
    return BR_OK;
}

int br_index_export_df_idf(const br_index* ix, int64_t* df_host, double* idf_host) {
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_index_export_df_idf: null handle");
    const size_t V = (size_t)ix->vocab;
    if (df_host) {
        if (ix->finalized) for (size_t t = 0; t < V; ++t) df_host[t] = ix->h_df_stat[t];
        else for (size_t t = 0; t < V; ++t) df_host[t] = (int64_t)ix->h_df[t];
    }
    if (idf_host) {
        BR_REQUIRE(ix->finalized, BR_ERR_STATE, "br_index_export_df_idf: idf needs br_index_finalize first");
        for (size_t t = 0; t < V; ++t) idf_host[t] = ix->h_idf[t];
    }
    return BR_OK;
}

int br_index_export_csr(const br_index* ix, int64_t* row_ptr_host, int32_t* doc_host, int32_t* tf_host,
                        int32_t* dl_host) {
    BR_REQUIRE(ix, BR_ERR_INVALID, "br_index_export_csr: null handle");
    BR_CUDA(cudaSetDevice(ix->device));
    if (row_ptr_host)
        BR_CUDA(cudaMemcpy(row_ptr_host, ix->row_ptr, sizeof(int64_t) * ((size_t)ix->vocab + 1), cudaMemcpyDeviceToHost));
    if (dl_host) BR_CUDA(cudaMemcpy(dl_host, ix->dl, sizeof(uint32_t) * (size_t)ix->n_docs, cudaMemcpyDeviceToHost));
    if ((doc_host || tf_host) && ix->nnz > 0) {
        BR_REQUIRE(doc_host && tf_host, BR_ERR_INVALID, "br_index_export_csr: doc_host and tf_host go together");
        br::DevArray<int32_t> d_doc, d_tf;
        BR_TRY(d_doc.alloc((size_t)ix->nnz));
        BR_TRY(d_tf.alloc((size_t)ix->nnz));
        br::k_export<<<br::blocks_for(ix->nnz, 256), 256>>>(ix->post, ix->tf, ix->nnz, d_doc, d_tf);
        BR_CUDA(cudaMemcpy(doc_host, d_doc, sizeof(int32_t) * (size_t)ix->nnz, cudaMemcpyDeviceToHost));
        BR_CUDA(cudaMemcpy(tf_host, d_tf, sizeof(int32_t) * (size_t)ix->nnz, cudaMemcpyDeviceToHost));
    }
    return BR_OK;
}

}  // extern "C"
