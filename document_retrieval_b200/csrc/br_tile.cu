// br_tile.cu - the fused BM25 path: doc-range tiled term-at-a-time scoring with the accumulators in shared memory
// and the top-k selection fused into the tile epilogue.
//
// Why: a dense [Q, N] fp32 accumulator costs 8 B x N of HBM traffic per query (zero + read back) and a global atomic
// per posting; at N = 8.8M that is more than the postings themselves (SURVEY 7, hard part 2).  Here a CTA owns (a tile
// of W x S consecutive docs) x (one query); each of its W = 8 warps owns one sub-range of S = 2^kSubShift = 2048 docs
// and walks, for the terms the query's plan streams, the slice of the term's posting list that falls in its sub-range
// (slice bounds come from the per-term skip table built with the index) and adds the packed fp32 weights into its
// private S accumulators: plain LDS/FFMA/STS, no atomics, no block barrier after the prologue, deterministic order.
// The accumulators are 64 KB per CTA (3 CTAs per SM).  Measured on the C4 workload with the same 64 KB split between
// queries and docs: 134k q/s at 4 queries x 512 docs, 150-164k at 2 x 1024, 185-191k at 1 x 2048 - a (query,
// sub-range) costs a fixed ~100 warp instructions of bookkeeping whatever it holds, and a 2048-doc slice of a rare term
// fills the 32 lanes of the walk where a 512-doc slice held 2-3 postings.
// The CTAs of all queries visit a tile back to back (blockIdx.x = query position), so the tile's posting slices come
// from HBM once per batch and from L2 afterwards.
//
// Terms too rare for a skip table ("cold": df < hot_min) are bucketed per batch instead: a counting sort of their
// postings by (tile, query) (k_cold_pass / scan); the CTA of a bucket adds those few entries with shared-memory atomics
// before its epilogue.
//
// Epilogue + selection: thr[q] is a lower bound of the k-th best fp32 score of query q over the shard (over the whole
// corpus with the cross-shard exchange).  A doc is emitted as a candidate iff score >= thr*(1-1e-5) (the band that
// makes the float64 re-score exact, see br_query.cu).  thr rises two ways: inside the kernel, when a sub-range holds k
// better docs in k different lanes (atomicMax); and between launches - tiles are processed in chunks of doubling size,
// and after each chunk k_tighten sets thr[q] to the k-th best score among the candidates emitted so far and compacts
// the list.  With doubling chunks every chunk emits about k new candidates per query, so the candidate list stays ~k
// long and the float64 re-score costs almost nothing.
#include <math_constants.h>

#include <algorithm>

#include <cub/cub.cuh>

#include "br_common.cuh"
#include "br_kernels.cuh"
#include "br_query.cuh"

namespace br {

constexpr int TILE_W = 8;            // warps per CTA = sub-ranges per tile
constexpr int TILE_SHIFT = kSubShift;         // docs per sub-range = 2^kSubShift (br_common.cuh; equals br_index::sub_shift)
constexpr int TILE_S = 1 << TILE_SHIFT;
constexpr int TILE_DOCS_SHIFT = TILE_SHIFT + 3;   // log2(W * S)
constexpr int TILE_QT = 20;          // max distinct hot terms of one query in the regular pass
constexpr int TILE_QT_LONG = 40;     // the same in the long-query pass (queries with up to 64 terms, e.g.
                                     // bigram-expanded queries, bm25_ranking.ipynb:105-107); more -> dense path
constexpr int TILE_CAP = 1024;       // candidates kept per query between tighten rounds (k <= 32)
// the same for 32 < k <= 1024: everything passes before the first threshold exists (the first launch covers TILE_CAP_BIG docs),
// later chunks add about k each
constexpr int TILE_CAP_BIG = (4 << kSubShift) > 8192 ? (4 << kSubShift) : 8192;
static_assert((1 << 3) == TILE_W, "TILE_DOCS_SHIFT assumes W == 8");
// tiles of the first launch (thresholds come from the seeding only): at most 32k docs, so that the docs passing a loose
// threshold fit the candidate list
constexpr int TILE_CHUNK0 = (32768 >> TILE_DOCS_SHIFT) >= 1 ? (32768 >> TILE_DOCS_SHIFT) : 1;
// Launch schedule and term classes; DESIGN.md 3.2 records other values of each within 1 % on the C4 workload.
constexpr int TILE_GROWTH = 2;       // every launch covers this many times the units of the one before
constexpr int TILE_TPB = 16;         // at most this many consecutive tiles per CTA (in the large launches)
constexpr int TILE_DENSE_MIN = 32;   // average postings of a term per sub-range from which its slices are walked
                                     // term by term (whole warp, pipelined) instead of by the sparse walk

struct __align__(16) TileEntry {
    int32_t term;
    int32_t slot;
    uint8_t mult;        // multiplicity of the term in the query
    uint8_t pos;         // index of the term in the query's unique-term list (bit of the query's deferral mask)
};

// a deferred term of one query: look-up row and multiplicity
struct __align__(8) NeEntry {
    int32_t row;
    float mult;
};
constexpr int NE_MAX = 32;           // deferred terms per query (a query on this path has <= 32 terms)

// cold entry: doc offset inside the tile (TILE_DOCS_SHIFT bits), weight
struct __align__(8) ColdEntry {
    uint32_t key;
    float w;
};

// ------------------------------------------------------------------------------------------
// query preparation: hot terms of each query, rows first, then dense postings, then sparse
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_tile_prep(PrepView pv, const int32_t* __restrict__ q_off,
                                                   const int32_t* __restrict__ hot_slot,
                                                   const int64_t* __restrict__ row_ptr, int32_t nq, int umax,
                                                   TileEntry* __restrict__ entries, int32_t* __restrict__ n_entries,
                                                   int32_t* __restrict__ elig, unsigned long long* __restrict__ cold_total,
                                                   int64_t dense_df_min, const int32_t* __restrict__ perm,
                                                   const int16_t* __restrict__ row_slot, int n_srows, int qt_max,
                                                   int max_terms) {
    __shared__ int32_t s_term[4][256];
    __shared__ uint8_t s_m[4][256], s_p[4][256];
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    const int g = blockIdx.x * 4 + wl;                   // query position
    if (g >= nq) return;
    const int q = perm[g];
    const int32_t off = q_off[q], nu = pv.u_cnt[q];
    int hot = 0, bad = 0;
    unsigned long long cold = 0;
    for (int base = 0; base < nu; base += 32) {
        const int j = base + lane;
        const int32_t t = j < nu ? pv.u_terms[off + j] : -1;
        const bool is_hot = t >= 0 && hot_slot[t] >= 0;
        if (t >= 0 && !is_hot) cold += (unsigned long long)(row_ptr[t + 1] - row_ptr[t]);
        if (t >= 0 && pv.u_mult[off + j] > 255) bad = 1;
        hot += __popc(__ballot_sync(0xffffffffu, is_hot));
    }
    for (int o = 16; o > 0; o >>= 1) cold += __shfl_xor_sync(0xffffffffu, cold, o);
    bad = __any_sync(0xffffffffu, bad);
    const bool ok = hot <= qt_max && !bad && pv.o_cnt[q] <= max_terms;   // longer queries: long pass / dense path
    if (lane == 0) elig[q] = ok ? 1 : 0;
    int n = 0;
    if (ok) {
        for (int base = 0; base < nu; base += 32) {
            const int j = base + lane;
            const int32_t t = j < nu ? pv.u_terms[off + j] : -1;
            const bool is_hot = t >= 0 && hot_slot[t] >= 0;
            const unsigned m = __ballot_sync(0xffffffffu, is_hot);
            if (is_hot) {
                const int p = n + __popc(m & ((1u << lane) - 1));
                s_term[wl][p] = t;
                s_m[wl][p] = (uint8_t)pv.u_mult[off + j];
                s_p[wl][p] = (uint8_t)j;
            }
            n += __popc(m);
        }
    }
    __syncwarp();
    // the query's hot terms (unique already), terms that are dense everywhere (df >= dense_df_min) first
    int U = 0, Ud = 0, Ur = 0;
    for (int pass = -1; pass < 2; ++pass) {
        for (int base = 0; base < n; base += 32) {
            const int i = base + lane;
            bool take = false;
            if (i < n) {
                const int32_t t = s_term[wl][i];
                const bool is_row = row_slot[t] >= 0 && row_slot[t] < n_srows;      // streamed row
                const bool dense = row_ptr[t + 1] - row_ptr[t] >= dense_df_min;
                const int cls = is_row ? -1 : (dense ? 0 : 1);          // rows first, then dense postings, then sparse
                take = cls == pass;
            }
            const unsigned m = __ballot_sync(0xffffffffu, take);
            if (take) {
                TileEntry e;
                e.term = s_term[wl][i];
                e.slot = pass < 0 ? (int32_t)row_slot[e.term] : hot_slot[e.term];
                e.mult = s_m[wl][i];
                e.pos = s_p[wl][i];
                entries[(int64_t)g * umax + U + __popc(m & ((1u << lane) - 1))] = e;
            }
            U += __popc(m);
        }
        if (pass < 0) Ur = U;
        if (pass == 0) Ud = U;
    }
    if (lane == 0) {
        n_entries[g] = U | (Ud << 10) | (Ur << 20);
        if (ok && cold) atomicAdd(cold_total, cold);
    }
}

// ------------------------------------------------------------------------------------------
// cold postings -> (tile, query position) buckets: counting sort
// ------------------------------------------------------------------------------------------
template <bool SCATTER>
__global__ void k_cold_pass(PrepView pv, const int32_t* __restrict__ q_off, const int32_t* __restrict__ hot_slot,
                            const int64_t* __restrict__ row_ptr, const br_posting* __restrict__ post, int32_t nq,
                            const int32_t* __restrict__ elig, const int32_t* __restrict__ inv_perm,
                            uint32_t* __restrict__ counter, ColdEntry* __restrict__ out, uint32_t out_cap) {
    const int lane = threadIdx.x & 31;
    const int q = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (q >= nq || !elig[q]) return;
    const int32_t off = q_off[q], nu = pv.u_cnt[q];
    const int g = inv_perm[q];
    for (int j = 0; j < nu; ++j) {
        const int32_t t = pv.u_terms[off + j];
        if (hot_slot[t] >= 0) continue;
        const float mult = (float)pv.u_mult[off + j];
        const int64_t lo = row_ptr[t], n = row_ptr[t + 1] - lo;
        for (int64_t i = lane; i < n; i += 32) {
            const br_posting p = post[lo + i];
            const uint32_t tile = p.doc >> TILE_DOCS_SHIFT;
            const int64_t b = (int64_t)tile * nq + g;
            const uint32_t pos = atomicAdd(counter + b, 1u);
            if (SCATTER && pos < out_cap) out[pos] = ColdEntry{p.doc & ((1u << TILE_DOCS_SHIFT) - 1), p.w * mult};
        }
    }
}

// three-kernel exclusive scan of uint32 counts (n up to ~2^31): out[i] = sum_{j<i} in[j], out[n] = total
constexpr int SCAN_T = 256, SCAN_I = 16, SCAN_TILE = SCAN_T * SCAN_I;
__global__ void __launch_bounds__(SCAN_T) k_scan_reduce(const uint32_t* __restrict__ in, int64_t n, uint32_t* __restrict__ part) {
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_I; ++j) {
        const int64_t i = base + j * SCAN_T + threadIdx.x;
        if (i < n) s += in[i];
    }
    uint32_t total;
    block_excl_scan(s, &total);
    if (threadIdx.x == 0) part[blockIdx.x] = total;
}
__global__ void __launch_bounds__(SCAN_T) k_scan_apply(const uint32_t* __restrict__ in, int64_t n,
                                                       const int64_t* __restrict__ part_off, uint32_t* __restrict__ out,
                                                       uint32_t* __restrict__ out_copy) {
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_I;
    uint32_t v[SCAN_I], s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_I; ++j) { v[j] = base + j < n ? in[base + j] : 0u; s += v[j]; }
    uint32_t total;
    uint32_t run = block_excl_scan(s, &total) + (uint32_t)part_off[blockIdx.x];
#pragma unroll
    for (int j = 0; j < SCAN_I; ++j) {
        if (base + j < n) { out[base + j] = run; out_copy[base + j] = run; }
        run += v[j];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == SCAN_T - 1) { out[n] = run; }
}

// ------------------------------------------------------------------------------------------
// the tile kernel
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sort_desc(float v, int lane) {
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const float o = __shfl_xor_sync(0xffffffffu, v, j);
            const bool up = (lane & k) == 0, lower = (lane & j) == 0;
            v = (lower == up) ? fmaxf(v, o) : fminf(v, o);
        }
    }
    return v;   // lane i holds the i-th largest
}


struct TileArgs {
    const br_posting* post;
    const int64_t* row_ptr;
    const uint32_t* skip;
    int32_t n_sub;
    int64_t n_docs;
    const TileEntry* entries;
    const int32_t* n_entries;
    int umax;
    int32_t nq;
    const int32_t* elig;
    const uint32_t* cold_off;     // [n_tiles * nq + 1] or null
    const ColdEntry* cold;
    uint32_t cold_cap;            // entries the cold buffer holds (a batch that needs more is repeated with a larger one)
    const float* rows;            // dense rows [n_rows, n_pad]
    int64_t n_pad;
    float* thr;
    int32_t* cand_cnt;
    int32_t* cand;                // [nq, cap]
    float* cand_h;                // [nq, cap]
    int cap;                      // candidate slots per query (TILE_CAP for k <= 32, TILE_CAP_BIG above)
    int K;
    int tile0;
    int tile_end;                 // tiles [tile0, tile_end) in this launch
    int sub_begin, sub_end;       // sub-ranges [sub_begin, sub_end) of those tiles (the large-k path starts with part of a tile)
    int tpb;                      // consecutive tiles per CTA
    int has_mult;                 // 0: every multiplicity is 1 (set(query) semantics)
    const int32_t* perm;          // position g -> query perm[g] (queries sorted by frequent-term signature)
    const uint32_t* defer_mask;   // [nq] bit j: the j-th unique term of the query is deferred in this launch
    const float* ne_ub;           // [nq] sum of the deferred terms' upper bounds (rounded up)
    const int16_t* row_slot;      // [V] look-up row of a term (every deferred term has one)
    // doc filter (k_tile_score<QT, true> only; appended so that the fields above keep their offsets)
    const uint32_t* fbits;        // bitmap rows [n_rows, fwords]
    int64_t fwords;
    const int32_t* frow;          // [nq] row of query qi, -1 = unfiltered
};

// the 4 docs doc .. doc+3 (doc a multiple of 4) of one lane share a bitmap word: zero the accumulators of the docs the
// filter excludes (they then neither pass the threshold nor raise it); docs >= n_docs are never read from the bitmap
__device__ __forceinline__ float4 filter4(float4 f, const uint32_t* fr, uint32_t doc, int64_t n_docs) {
    if (!fr) return f;
    const uint32_t b = (int64_t)doc < n_docs ? (__ldg(fr + (doc >> 5)) >> (doc & 31)) : 0u;
    f.x = (b & 1u) ? f.x : 0.f;
    f.y = (b & 2u) ? f.y : 0.f;
    f.z = (b & 4u) ? f.z : 0.f;
    f.w = (b & 8u) ? f.w : 0.f;
    return f;
}

constexpr int SPX = 1;               // postings per lane requested ahead for a sparse slice (2 was measured no faster)
constexpr int LIST_CAP = 64;         // crossing-list slots per warp and sub-range (overflow -> full scan of the sub-range)

// MaxScore deferral (exact): between launches every query gets a plan (make_plan): the terms with the smallest upper
// bounds ub[t] = max posting weight, as long as their sum stays below a fraction of the query's threshold, are
// "deferred" - not streamed at all.  A doc whose partial score p over the streamed ("essential") terms satisfies
// p + sum(deferred ub) < thr*(1-band) cannot reach the threshold and is never looked at; the few others are completed
// by direct look-ups before the usual filter: every deferrable term (df >= N/64) has a look-up row w[row][doc], so a
// completion is a handful of independent 4-byte loads, no search.  The densest terms have the smallest bounds, so in
// the steady state neither the streamed rows nor the dense posting slices are read.
// Without streamed rows every accumulator starts at zero and only grows, so the lane that has just updated one knows
// whether it has reached t1 = thr*(1-band) - sum(deferred ub): it records the doc in its warp's crossing list, and
// after the posting phases the warp completes and filters just the listed docs (an atomic exchange on the accumulator
// removes duplicates).  The S accumulators of a sub-range are scanned only when the query still streams rows / has no
// threshold yet, or when the crossing list overflows.
// After the CTA prologue there is no block barrier: every warp fetches the slice bounds of its own sub-range (one tile
// ahead, into registers) and its own copy of the threshold.
// FILT (filtered batches): a doc the query's filter row excludes is never emitted and never raises the threshold - the
// crossing list tests its bit before the completion, the scan epilogue zeroes its accumulator - so every threshold stays
// the score of k distinct ALLOWED docs, a valid lower bound of the filtered k-th best score.
template <int QT, bool FILT>
__global__ void __launch_bounds__(TILE_W * 32, 3) k_tile_score(TileArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* acc = reinterpret_cast<float*>(smem_raw);                                     // [W][S]
    TileEntry* ent = reinterpret_cast<TileEntry*>(smem_raw + sizeof(float) * TILE_W * TILE_S);   // streamed entries
    int64_t* s_base = reinterpret_cast<int64_t*>(ent + a.umax);                          // [umax]
    float* s_fm = reinterpret_cast<float*>(s_base + a.umax);                             // [umax] multiplicities as floats
    uint32_t* s_skiprow = reinterpret_cast<uint32_t*>(s_fm + a.umax);                    // [umax] slot * (n_sub+1)
    NeEntry* s_ne = reinterpret_cast<NeEntry*>(s_skiprow + a.umax);                      // [NE_MAX] deferred terms
    uint2* s_bnd_all = reinterpret_cast<uint2*>(s_ne + NE_MAX);                          // [W][umax] slice (lo, hi) per warp
    uint16_t* s_list_all = reinterpret_cast<uint16_t*>(s_bnd_all + TILE_W * a.umax);     // [W][LIST_CAP]
    // small per-CTA / per-warp state, carved from the same buffer (static __shared__ arrays would have their window
    // addresses rematerialised all over the kernel)
    int* s_cnt = reinterpret_cast<int*>(s_list_all + TILE_W * LIST_CAP);                 // Ur, Ud, U (streamed), rows, deferred
                                                                                         // terms (padded to x4), sparse terms
    int* s_lcnt_all = s_cnt + 6;                                                         // [W]
    uint8_t* s_ql_all = reinterpret_cast<uint8_t*>(s_lcnt_all + TILE_W);                 // [W][umax] non-empty sparse slices

    const int g = blockIdx.x;                                           // query position
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int tile_first = a.tile0 + blockIdx.y * a.tpb;
    const int tile_last = min(tile_first + a.tpb, a.tile_end);          // exclusive
    const int qi = a.perm[g];
    if (!a.elig[qi]) return;                                            // served by the long pass / the dense path
    const float neub = a.ne_ub[qi];
    const uint32_t* frow = nullptr;                                     // the query's filter row (nullptr: unfiltered)
    if constexpr (FILT) frow = a.frow[qi] >= 0 ? a.fbits + (int64_t)a.frow[qi] * a.fwords : nullptr;

    if (w == 0) {
        // split the query's entries into streamed and deferred ones (stable: rows, dense postings, sparse)
        const int U0 = a.n_entries[g] & 0x3ff, Ud0 = (a.n_entries[g] >> 10) & 0x3ff, Ur0 = a.n_entries[g] >> 20;
        const uint32_t dm = a.defer_mask[qi];
        int na = 0, ur = 0, ud = 0, nne = 0;
        bool rows = false;
        for (int base = 0; base < U0; base += 32) {
            const int u = base + lane;
            TileEntry e{};
            float act = 0.f, def = 0.f;
            if (u < U0) {
                e = a.entries[(int64_t)g * a.umax + u];
                if (e.pos < 32 && ((dm >> e.pos) & 1u)) def = (float)e.mult;
                else { act = (float)e.mult; if (u < Ur0) rows = true; }
            }
            const bool isa = act != 0.f;
            const unsigned ma = __ballot_sync(0xffffffffu, isa);
            const unsigned lt = (1u << lane) - 1;
            if (isa) {
                const int p = na + __popc(ma & lt);
                ent[p] = e;
                s_base[p] = a.row_ptr[e.term];
                s_fm[p] = act;
                s_skiprow[p] = (uint32_t)e.slot * (uint32_t)(a.n_sub + 1);      // row terms: slot = row index (unused here)
            }
            const unsigned md = __ballot_sync(0xffffffffu, def != 0.f);          // list of deferred terms
            if (def != 0.f) {
                const int p = nne + __popc(md & lt);
                if (p < NE_MAX) s_ne[p] = NeEntry{(int32_t)a.row_slot[e.term], def};
            }
            nne += __popc(md);
            ur += __popc(ma & __ballot_sync(0xffffffffu, u < Ur0));
            ud += __popc(ma & __ballot_sync(0xffffffffu, u < Ud0));
            na += __popc(ma);
        }
        rows = __any_sync(0xffffffffu, rows);
        const int n = min(nne, NE_MAX), n4 = (n + 3) & ~3;
        if (lane >= n && lane < n4) s_ne[lane] = NeEntry{0, 0.f};     // padding: row 0, multiplicity 0
        if (lane == 0) { s_cnt[0] = ur; s_cnt[1] = ud; s_cnt[2] = na; s_cnt[3] = rows ? 1 : 0; s_cnt[4] = n4; }
    }
    __syncthreads();                                   // the only block barrier: from here on the warps run independently
    const int Ur = s_cnt[0], Ud = s_cnt[1], U = s_cnt[2];
    const bool rows = s_cnt[3] != 0;
    const int nne = s_cnt[4];
    uint2* s_bnd = s_bnd_all + w * a.umax;
    uint8_t* s_ql = s_ql_all + w * a.umax;
    uint16_t* s_list = s_list_all + w * LIST_CAP;
    int* s_lcnt = s_lcnt_all + w;

    // slice bounds of this warp's sub-range: lane covers entries lane, lane+32, ...; fetched one tile ahead
    constexpr int NR = (QT + 31) / 32;
    uint32_t nlo[NR], nhi[NR];
    auto load_bounds = [&](int sub) {
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int u = lane + 32 * r;
            nlo[r] = nhi[r] = 0;
            if (u >= Ur && u < U) {
                const uint32_t* sk = a.skip + s_skiprow[u] + sub;
                nlo[r] = __ldg(sk);
                nhi[r] = __ldg(sk + 1);
            }
        }
    };
    // stores the bounds and lists the sparse entries whose slice in this sub-range is not empty (entry order kept);
    // returns their number
    auto store_bounds = [&]() {
        int n = 0;
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const int u = lane + 32 * r;
            if (u < U) s_bnd[u] = make_uint2(nlo[r], nhi[r]);     // row terms keep empty slices
            const bool sp = u >= Ud && u < U && nlo[r] < nhi[r];
            const unsigned m = __ballot_sync(0xffffffffu, sp);
            if (sp) s_ql[n + __popc(m & ((1u << lane) - 1u))] = (uint8_t)u;
            n += __popc(m);
        }
        return n;
    };
    // (large-k path: a launch may start inside its first tile - the warps below sub_begin start one tile later)
    const int tile_begin_w = tile_first + ((tile_first * TILE_W + w < a.sub_begin) ? 1 : 0);
    if (tile_begin_w * TILE_W + w < a.n_sub) load_bounds(tile_begin_w * TILE_W + w);
#pragma unroll 1
    for (int tile = tile_begin_w; tile < tile_last; ++tile) {
    const int sub = tile * TILE_W + w;
    if (sub >= a.sub_end) break;                                      // warp-uniform; the later tiles are out of range too
    const int nql = store_bounds();
    if (tile + 1 < tile_last && sub + TILE_W < a.n_sub) load_bounds(sub + TILE_W);     // in flight during this tile
    // threshold of this tile (a stale, lower value is always valid); t1: partial scores below it cannot reach thr.
    // A query that is scanned anyway (streamed rows / no threshold yet) never pushes: its t1 is +inf.
    float th = 0.f;
    if (lane == 0) th = __ldcg(a.thr + qi);
    th = __shfl_sync(0xffffffffu, th, 0);
    const float t = th * (1.f - kBandRel) * (1.f - kBandRel) - neub;
    const float t1 = (rows || !(t > 0.f)) ? CUDART_INF_F : t;
    bool scan = t1 == CUDART_INF_F;
    if (lane == 0) *s_lcnt = 0;
    // bucket bounds of this (tile, query)'s cold postings: requested here, used after the posting phases
    uint32_t cold0 = 0, cold1 = 0;
    if (a.cold_off) {
        const uint32_t* co = a.cold_off + ((int64_t)tile * a.nq + g);
        cold0 = __ldg(co);
        cold1 = __ldg(co + 1);
    }
    __syncwarp();
    const uint32_t doc0 = (uint32_t)sub << TILE_SHIFT;
    float* my = acc + w * TILE_S;
    auto push = [&](uint32_t idx) {                     // record a crossing (rare)
        const int p = atomicAdd(s_lcnt, 1);
        if (p < LIST_CAP) s_list[p] = (uint16_t)idx;
    };
    if (Ur == 0) {
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int s4 = 0; s4 < TILE_S / 128; ++s4) reinterpret_cast<float4*>(my)[s4 * 32 + lane] = z;
    } else {
        // each warp initialises its own accumulators: zero + the weights of the streamed dense-row terms (terms present
        // in >= ~20% of the docs are stored as plain fp32 rows, 0 where absent), 4 docs per lane
#pragma unroll 1
        for (int seg = 0; seg < TILE_S / 128; ++seg) {          // 128 docs per pass
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int64_t off = (int64_t)doc0 + seg * 128 + lane * 4;
            for (int u0 = 0; u0 < Ur; u0 += 2) {             // two rows in flight
                float4 d[2];
                float ff[2];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int u = min(u0 + k, Ur - 1);
                    d[k] = __ldg(reinterpret_cast<const float4*>(a.rows + (int64_t)ent[u].slot * a.n_pad + off));
                    ff[k] = u0 + k < Ur ? s_fm[u] : 0.f;
                }
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    if (ff[k] != 0.f) {                      // warp-uniform
                        v.x = fmaf(d[k].x, ff[k], v.x);
                        v.y = fmaf(d[k].y, ff[k], v.y);
                        v.z = fmaf(d[k].z, ff[k], v.z);
                        v.w = fmaf(d[k].w, ff[k], v.w);
                    }
                }
            }
            reinterpret_cast<float4*>(my)[seg * 32 + lane] = v;
        }
    }
    __syncwarp();

    // Phase A - sparse slices (most (term, sub-range) pairs hold 0-8 postings): the warp walks the list of the
    // sub-range's non-empty sparse slices straight from shared memory - slice bounds, list base and multiplicity of slice
    // i are broadcast reads, the postings of slice i+1 are requested before slice i is added.  (Pulling the next non-empty slice over by shuffle from the lane
    // that fetched its bounds cost three shuffles, a find-first-set and two votes per step and was slower: DESIGN.md 3.2.)
    {
        const uint2* const post2 = reinterpret_cast<const uint2*>(a.post);
        uint32_t c_hi = 0, c_lo = 0, c_pb = 0;
        float c_mu = 1.f;
        uint2 c_p[SPX];
        auto fetch = [&](int it, uint32_t& lo, uint32_t& hi, uint32_t& pb, float& mu, uint2* p) {
            lo = hi = 0;
            if (it < nql) {
                const int u = s_ql[it];
                const uint2 bd = s_bnd[u];
                lo = bd.x; hi = bd.y;
                pb = (uint32_t)s_base[u];                           // posting index of the term's list (nnz < 2^32)
                if (a.has_mult) mu = s_fm[u];
#pragma unroll
                for (int x = 0; x < SPX; ++x)
                    if (lo + 32 * x + lane < hi) p[x] = __ldg(post2 + pb + lo + 32 * x + lane);
            }
        };
        fetch(0, c_lo, c_hi, c_pb, c_mu, c_p);
#pragma unroll 1
        for (int it = 0; it < nql; ++it) {
            uint32_t n_lo, n_hi, n_pb = 0;
            float n_mu = 1.f;
            uint2 n_p[SPX];
            fetch(it + 1, n_lo, n_hi, n_pb, n_mu, n_p);
#pragma unroll
            for (int x = 0; x < SPX; ++x) {
                if (c_lo + 32 * x + lane < c_hi) {                  // one term: distinct docs
                    const uint32_t idx = c_p[x].x - doc0;
                    const float val = fmaf(__uint_as_float(c_p[x].y), c_mu, my[idx]);
                    my[idx] = val;
                    if (val >= t1) push(idx);
                }
            }
            // a slice longer than the postings fetched ahead
            for (uint32_t c = c_lo + 32 * SPX; __any_sync(0xffffffffu, c < c_hi); c += 32) {
                __syncwarp();
                if (c + lane < c_hi) {
                    const uint2 p = __ldg(post2 + c_pb + c + lane);
                    const uint32_t idx = p.x - doc0;
                    const float val = fmaf(__uint_as_float(p.y), c_mu, my[idx]);
                    my[idx] = val;
                    if (val >= t1) push(idx);
                }
            }
            __syncwarp();
            c_lo = n_lo; c_hi = n_hi; c_pb = n_pb; c_mu = n_mu;
#pragma unroll
            for (int x = 0; x < SPX; ++x) c_p[x] = n_p[x];
        }
    }
    __syncwarp();
    // Phase B - dense slices (terms with >= TILE_DENSE_MIN postings per sub-range on average that are still streamed:
    // rare once the deferral plans exist), 64 postings per step.  Inside a term all docs are distinct, so the
    // read-modify-writes of a step are independent.  No atomics.
#pragma unroll 1
    for (int u = Ur; u < Ud; ++u) {
        const uint2 bd = s_bnd[u];
        if (bd.x >= bd.y) continue;
        const float ff = s_fm[u];
        const uint2* p = reinterpret_cast<const uint2*>(a.post) + s_base[u];
        // the next 64 postings are requested before the current 64 are added (ncu: 10 % of the stall samples of the
        // 2048-doc version sat on the first use of an unprefetched chunk)
        uint2 nv2[2];
#pragma unroll
        for (int x = 0; x < 2; ++x) {
            nv2[x] = make_uint2(0xffffffffu, 0u);
            if (bd.x + lane + 32 * x < bd.y) nv2[x] = __ldg(p + bd.x + lane + 32 * x);
        }
        for (uint32_t c = bd.x; c < bd.y; c += 64) {
            uint2 v[2];
#pragma unroll
            for (int x = 0; x < 2; ++x) {
                v[x] = nv2[x];
                nv2[x] = make_uint2(0xffffffffu, 0u);
                if (c + 64 + lane + 32 * x < bd.y) nv2[x] = __ldg(p + c + 64 + lane + 32 * x);
            }
#pragma unroll
            for (int x = 0; x < 2; ++x) {
                if (v[x].x != 0xffffffffu) {
                    const uint32_t idx = v[x].x - doc0;
                    const float nv = fmaf(__uint_as_float(v[x].y), ff, my[idx]);
                    my[idx] = nv;
                    if (nv >= t1) push(idx);
                }
            }
        }
    }
    __syncwarp();
    // cold postings of this (tile, query) bucket that fall in this warp's sub-range
    if (a.cold_off) {
        const uint32_t c0 = cold0, c1 = min(cold1, a.cold_cap);
        for (uint32_t i = c0 + lane; i < c1; i += 32) {
            const ColdEntry ce = a.cold[i];
            if ((ce.key >> TILE_SHIFT) == (uint32_t)w) {
                const uint32_t idx = ce.key & (TILE_S - 1);
                const float nv = atomicAdd(my + idx, ce.w) + ce.w;
                if (nv >= t1) push(idx);
            }
        }
    }
    __syncwarp();

    // crossing list: complete (deferred terms by look-up row) and filter exactly the listed docs, one per lane
    const int n_list = *s_lcnt;
    if (n_list > LIST_CAP) {
        scan = true;                                                   // overflow: scan the sub-range instead
    } else {
        for (int i0 = 0; i0 < n_list; i0 += 32) {
            const int i = i0 + lane;
            if (i < n_list) {
                const uint32_t idx = s_list[i];
                // a doc is listed once per update at or above t1: the first taker marks the accumulator
                float full = atomicExch(my + idx, -1.f);
                bool live = full > 0.f;
                if constexpr (FILT) live = live && doc_allowed(frow, doc0 + idx);
                if (live) {
                    const float* col = a.rows + (doc0 + idx);
                    for (int x0 = 0; x0 < nne; x0 += 4) {          // lists are padded to a multiple of 4
                        float wv[4], mm[4];
#pragma unroll
                        for (int x = 0; x < 4; ++x) {
                            const NeEntry e2 = s_ne[x0 + x];
                            mm[x] = e2.mult;
                            wv[x] = __ldg(col + (int64_t)e2.row * a.n_pad);
                        }
#pragma unroll
                        for (int x = 0; x < 4; ++x) full = fmaf(wv[x], mm[x], full);
                    }
                    if (full >= th * (1.f - kBandRel)) {
                        const int pos = atomicAdd(a.cand_cnt + qi, 1);
                        if (pos < a.cap) {
                            a.cand[(int64_t)qi * a.cap + pos] = (int32_t)(doc0 + idx);
                            a.cand_h[(int64_t)qi * a.cap + pos] = full;
                        }
                    }
                }
            }
        }
    }
    __syncwarp();

    // scan epilogue: threshold filter over all S accumulators of the sub-range (streamed rows, no threshold yet, overflow)
    auto scan_epilogue = [&]() {
        float v[TILE_S / 32];                                   // v[4*s + e] = doc s*128 + lane*4 + e
        float mx = 0.f;
#pragma unroll
        for (int s = 0; s < TILE_S / 128; ++s) {
            float4 f = reinterpret_cast<const float4*>(my)[s * 32 + lane];
            if constexpr (FILT) f = filter4(f, frow, doc0 + s * 128 + lane * 4, a.n_docs);
            v[4 * s + 0] = f.x; v[4 * s + 1] = f.y; v[4 * s + 2] = f.z; v[4 * s + 3] = f.w;
            mx = fmaxf(fmaxf(mx, fmaxf(f.x, f.y)), fmaxf(f.z, f.w));
        }
        if (!__any_sync(0xffffffffu, mx >= t && mx > 0.f)) return;        // nothing can reach the threshold here
        float lo_thr = th * (1.f - kBandRel);
        if (nne > 0) {
            // (overflow path) complete the partial scores that may still reach the threshold, in place
            static_assert(TILE_S / 32 <= 64, "completion mask of the scan epilogue: one bit per doc of a lane");
            unsigned long long pm = 0;
#pragma unroll
            for (int j = 0; j < TILE_S / 32; ++j) pm |= (v[j] >= t && v[j] > 0.f) ? (1ull << j) : 0ull;
            while (pm) {
                const int j = __ffsll((long long)pm) - 1;
                pm &= pm - 1;
                const uint32_t idx = (uint32_t)((j >> 2) * 128 + lane * 4 + (j & 3));
                const float* col = a.rows + (doc0 + idx);
                float full = my[idx];
                for (int i = 0; i < nne; ++i) full = fmaf(__ldg(col + (int64_t)s_ne[i].row * a.n_pad), s_ne[i].mult, full);
                my[idx] = full;
            }
            __syncwarp();
            mx = 0.f;
#pragma unroll
            for (int s = 0; s < TILE_S / 128; ++s) {
                float4 f = reinterpret_cast<const float4*>(my)[s * 32 + lane];
                if constexpr (FILT) f = filter4(f, frow, doc0 + s * 128 + lane * 4, a.n_docs);
                v[4 * s + 0] = f.x; v[4 * s + 1] = f.y; v[4 * s + 2] = f.z; v[4 * s + 3] = f.w;
                mx = fmaxf(fmaxf(mx, fmaxf(f.x, f.y)), fmaxf(f.z, f.w));
            }
        }
        int c = 0;
#pragma unroll
        for (int j = 0; j < TILE_S / 32; ++j) c += (v[j] >= lo_thr && v[j] > 0.f) ? 1 : 0;
        int tot = c;
        for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
        if (tot == 0) return;
        if (tot >= a.K && a.K <= 32) {
            // K distinct docs (one per lane) score >= the K-th largest lane maximum: a valid lower
            // bound of the K-th best score of this query over the whole shard (a lane maximum that is only a
            // partial score is a lower bound of that doc's score, so the bound stays valid)
            const float srt = warp_sort_desc(mx, lane);
            const float kth = __shfl_sync(0xffffffffu, srt, a.K - 1);
            if (kth > th) {
                th = kth;
                if (lane == 0) atomicMax(reinterpret_cast<int*>(a.thr + qi), __float_as_int(kth));   // scores >= 0
                lo_thr = th * (1.f - kBandRel);
                c = 0;
#pragma unroll
                for (int j = 0; j < TILE_S / 32; ++j) c += (v[j] >= lo_thr && v[j] > 0.f) ? 1 : 0;
            }
        }
        // warp-exclusive offsets, one global atomic per sub-range
        int incl = c;
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0) return;
        int base = 0;
        if (lane == 0) base = atomicAdd(a.cand_cnt + qi, total);
        base = __shfl_sync(0xffffffffu, base, 0);
        int pos = base + incl - c;
        int32_t* out = a.cand + (int64_t)qi * a.cap;
        float* out_h = a.cand_h + (int64_t)qi * a.cap;
#pragma unroll
        for (int j = 0; j < TILE_S / 32; ++j) {
            if (v[j] >= lo_thr && v[j] > 0.f) {
                if (pos < a.cap) { out[pos] = (int32_t)(doc0 + (j >> 2) * 128 + lane * 4 + (j & 3)); out_h[pos] = v[j]; }
                ++pos;
            }
        }
    };
    if (scan) scan_epilogue();
    __syncwarp();
    }   // tile loop
}

// Deferral plan of one query for the next launch (one warp; see k_tile_score): greedily defer the hot terms with the
// smallest upper bound mult * ub[t] while their sum stays below frac * thr * (1 - band).  Cold terms (no skip table)
// are never deferred.  ne_ub is rounded up so that "partial + ne_ub < t" really excludes the doc.
struct PlanArgs {
    const int32_t* q_off;
    const int32_t* u_terms;
    const int32_t* u_mult;
    const int32_t* u_cnt;
    const float* ub;
    const int16_t* row_slot;
    int n_srows;
    float frac;
    uint32_t* defer_mask;
    float* ne_ub;
};
// Only terms with a look-up row can be deferred.  The streamed-row terms (the densest, smallest bounds) go first and
// all of them or nothing: a query whose accumulators start from rows needs the full epilogue scan anyway.
__device__ __forceinline__ void make_plan(const PlanArgs& pa, int q, float thr, int lane) {
    const int32_t off = pa.q_off[q], nu = pa.u_cnt[q];
    uint32_t mask = 0;
    float sum = 0.f;
    if (thr > 0.f && pa.frac > 0.f && nu <= 32) {
        float v = CUDART_INF_F;
        bool srow = false;
        if (lane < nu) {
            const int32_t t = pa.u_terms[off + lane];
            const int rs = pa.row_slot[t];
            if (rs >= 0) { v = pa.ub[t] * (float)pa.u_mult[off + lane]; srow = rs < pa.n_srows; }
        }
        const float budget = thr * (1.f - kBandRel) * pa.frac;
        float ssum = srow ? v : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ssum += __shfl_xor_sync(0xffffffffu, ssum, o);
        if (ssum < budget) {
            mask = __ballot_sync(0xffffffffu, srow);
            sum = ssum;
            if (srow) v = CUDART_INF_F;
            for (int it = 0; it < nu; ++it) {
                float best = v;
                int who = lane;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
                    const int ow = __shfl_xor_sync(0xffffffffu, who, o);
                    if (ob < best || (ob == best && ow < who)) { best = ob; who = ow; }
                }
                if (!(sum + best < budget)) break;         // also stops at +inf (nothing deferrable left)
                sum += best;
                mask |= 1u << who;
                if (lane == who) v = CUDART_INF_F;
            }
        }
    }
    if (lane == 0) {
        pa.defer_mask[q] = mask;
        pa.ne_ub[q] = sum * (1.f + 1e-6f);
    }
}

// Threshold seeding (K <= 32): before any tile is scored, thr[q] := the largest, over the query's terms with df >= K,
// of the K-th largest weight among the term's first SEED_MAX postings - K distinct docs score at least that much, so it
// is a valid lower bound of the K-th best score, and the first launches already run with a deferral plan instead of
// streaming every term against a zero threshold.  One warp per query; a running top-32 is kept sorted across the lanes
// (each batch of 32 weights is sorted, reversed and merged bitonically).
// Only the postings of docs the query's filter row allows count (K distinct ALLOWED docs score at least the seed).
constexpr int SEED_MAX = 256;
__global__ void __launch_bounds__(128) k_seed_thr(const br_posting* __restrict__ post, const int64_t* __restrict__ row_ptr,
                                                  int32_t nq, int K, const int32_t* __restrict__ elig, float* __restrict__ thr,
                                                  PlanArgs pa, DocFilter f) {
    const int lane = threadIdx.x & 31;
    const int q = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (q >= nq || !elig[q]) return;
    const uint32_t* fr = f.row ? f.row_of(q) : nullptr;
    const int32_t off = pa.q_off[q], nu = pa.u_cnt[q];
    float best = 0.f;
    for (int j = nu - 1; j >= 0; --j) {         // descending term id: in a frequency-ranked vocabulary the rare (high-bound)
        const int32_t t = pa.u_terms[off + j];  // terms come first and the frequent ones are then skipped by the ub test
        const float m = (float)pa.u_mult[off + j];
        const int64_t lo = row_ptr[t], df = row_ptr[t + 1] - lo;
        if (df < K || !(pa.ub[t] * m > best)) continue;            // cannot raise the bound
        const int n = (int)min(df, (int64_t)SEED_MAX);
        float run = 0.f;                                            // lane i: i-th largest weight so far
        for (int base = 0; base < n; base += 32) {
            const float wv = base + lane < n && doc_allowed(fr, post[lo + base + lane].doc) ? post[lo + base + lane].w * m : 0.f;
            const float srt = warp_sort_desc(fmaxf(wv, 0.f), lane);
            float x = fmaxf(run, __shfl_sync(0xffffffffu, srt, 31 - lane));     // bitonic: top 32 of the union
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float y = __shfl_xor_sync(0xffffffffu, x, o);
                x = (lane & o) ? fminf(x, y) : fmaxf(x, y);
            }
            run = x;
        }
        best = fmaxf(best, __shfl_sync(0xffffffffu, run, K - 1));
    }
    const float th = best * (1.f - 4e-6f);      // fp32 accumulation of the doc's other terms can only add; slack for rounding
    if (lane == 0) thr[q] = th;
    make_plan(pa, q, th, lane);
}

// Between chunks: thr[q] = max(thr[q], K-th best fp32 score emitted so far); keep only the candidates
// inside the band of the new threshold (sorted by score); sticky overflow flag.
constexpr int TG_T = 256, TGS_T = 64;
__global__ void __launch_bounds__(TGS_T) k_tighten(float* __restrict__ thr, int32_t* __restrict__ cand_cnt,
                                                  int32_t* __restrict__ prev_cnt, int32_t* __restrict__ cand,
                                                  float* __restrict__ cand_h, int K, int32_t* __restrict__ overflow,
                                                  PlanArgs pa) {
    __shared__ float s_h[TILE_CAP];
    __shared__ int32_t s_id[TILE_CAP];
    __shared__ int s_keep;
    const int q = blockIdx.x;
    int n = cand_cnt[q];
    if (n == prev_cnt[q]) return;                      // nothing emitted since the last round
    if (n > TILE_CAP) {
        if (threadIdx.x == 0) overflow[q] = 1;
        n = TILE_CAP;
    }
    int32_t* ids = cand + (int64_t)q * TILE_CAP;
    float* hs = cand_h + (int64_t)q * TILE_CAP;
    int n_sort = 32;                                   // smallest power of two covering the list
    while (n_sort < n) n_sort <<= 1;
    for (int i = threadIdx.x; i < n_sort; i += TGS_T) {
        s_h[i] = i < n ? hs[i] : -1.f;
        s_id[i] = i < n ? ids[i] : -1;
    }
    if (threadIdx.x == 0) s_keep = 0;
    for (int size = 2; size <= n_sort; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < n_sort / 2; i += TGS_T) {
                const int x = 2 * i - (i & (stride - 1)), y = x + stride;
                const bool up = (x & size) == 0;
                const float hx = s_h[x], hy = s_h[y];
                if ((hy > hx) == up) {
                    s_h[x] = hy; s_h[y] = hx;
                    const int32_t t = s_id[x]; s_id[x] = s_id[y]; s_id[y] = t;
                }
            }
        }
    }
    __syncthreads();
    float th = thr[q];
    if (n >= K && s_h[K - 1] > th) th = s_h[K - 1];
    const float lo = th * (1.f - kBandRel);
    int keep = 0;
    for (int i = threadIdx.x; i < n; i += TGS_T) keep += (s_h[i] >= lo) ? 1 : 0;
    for (int o = 16; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    if ((threadIdx.x & 31) == 0 && keep) atomicAdd(&s_keep, keep);
    __syncthreads();
    keep = s_keep;
    for (int i = threadIdx.x; i < n; i += TGS_T) {
        ids[i] = i < keep ? s_id[i] : -1;
        hs[i] = i < keep ? s_h[i] : 0.f;
    }
    if (threadIdx.x == 0) {
        thr[q] = th;
        cand_cnt[q] = keep;
        prev_cnt[q] = keep;
    }
    if (threadIdx.x < 32) make_plan(pa, q, th, threadIdx.x);
}

// The same for long candidate lists (32 < K <= 1024, up to TILE_CAP_BIG entries): the K-th largest score by a 4 x 8-bit
// radix select over the list in shared memory (scores are positive floats, so their bit patterns order like integers)
// instead of a sort; survivors (score >= new threshold x (1 - band)) are compacted to the head of the query's region in
// arbitrary order - every survivor is re-scored in float64 and ordered by k_final_select afterwards.
__global__ void __launch_bounds__(TG_T) k_tighten_big(float* __restrict__ thr, int32_t* __restrict__ cand_cnt,
                                                      int32_t* __restrict__ prev_cnt, int32_t* __restrict__ cand,
                                                      float* __restrict__ cand_h, int K, int cap, int scap,
                                                      int32_t* __restrict__ overflow, PlanArgs pa) {
    // scap <= cap: list entries the shared-memory copy holds in this round (the whole region after the first launch,
    // which can pass a full tile; half of it later, when the lists are ~K long - a longer one goes to the dense path)
    extern __shared__ __align__(16) unsigned char tb_smem[];
    uint32_t* s_h = reinterpret_cast<uint32_t*>(tb_smem);             // [scap] score bits
    int32_t* s_id = reinterpret_cast<int32_t*>(s_h + scap);           // [scap]
    __shared__ uint32_t s_hist[256];
    __shared__ uint32_t s_prefix, s_need;
    const int q = blockIdx.x;
    int n = cand_cnt[q];
    if (n == prev_cnt[q]) return;                      // nothing emitted since the last round
    if (n > scap) {
        if (threadIdx.x == 0) overflow[q] = 1;
        n = scap;
    }
    int32_t* ids = cand + (int64_t)q * cap;
    float* hs = cand_h + (int64_t)q * cap;
    for (int i = threadIdx.x; i < n; i += TG_T) {
        s_h[i] = __float_as_uint(hs[i]);
        s_id[i] = ids[i];
    }
    float th = thr[q];
    if (n >= K) {
        if (threadIdx.x == 0) { s_prefix = 0; s_need = (uint32_t)K; }
        for (int shift = 24; shift >= 0; shift -= 8) {
            s_hist[threadIdx.x] = 0;                  // TG_T == 256 bins
            __syncthreads();
            const uint32_t prefix = s_prefix, need = s_need;
            const uint32_t himask = shift == 24 ? 0u : (0xffffffffu << (shift + 8));
            for (int i = threadIdx.x; i < n; i += TG_T) {
                const uint32_t b = s_h[i];
                if ((b & himask) == prefix) atomicAdd(&s_hist[(b >> shift) & 0xff], 1u);
            }
            __syncthreads();
            if (threadIdx.x == 0) {                   // walk the bins from the top until `need` elements are covered
                uint32_t acc = 0;
                int b = 255;
                for (; b > 0; --b) {
                    if (acc + s_hist[b] >= need) break;
                    acc += s_hist[b];
                }
                s_prefix = prefix | ((uint32_t)b << shift);
                s_need = need - acc;
            }
            __syncthreads();
        }
        const float kth = __uint_as_float(s_prefix);  // exactly the K-th largest score of the list
        if (kth > th) th = kth;
    }
    __syncthreads();
    const uint32_t lo = __float_as_uint(th * (1.f - kBandRel));
    // stable compaction in rounds of TG_T elements
    __shared__ int s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += TG_T) {
        const int i = i0 + threadIdx.x;
        const bool keep = i < n && s_h[i] >= lo;
        uint32_t total;
        const uint32_t ex = block_excl_scan(keep ? 1u : 0u, &total);
        const int base = s_base;
        if (keep) {
            ids[base + ex] = s_id[i];
            hs[base + ex] = __uint_as_float(s_h[i]);
        }
        __syncthreads();
        if (threadIdx.x == 0) s_base = base + (int)total;
        __syncthreads();
    }
    const int kept = s_base;
    for (int i = kept + threadIdx.x; i < n; i += TG_T) {
        ids[i] = -1;
        hs[i] = 0.f;
    }
    if (threadIdx.x == 0) {
        thr[q] = th;
        cand_cnt[q] = kept;
        prev_cnt[q] = kept;
    }
    if (threadIdx.x < 32) make_plan(pa, q, th, threadIdx.x);
}

__global__ void k_fused_flags(const int32_t* __restrict__ elig, const int32_t* __restrict__ overflow,
                              const int32_t* __restrict__ out_cnt, int32_t nq, int32_t need, int positive_only,
                              int32_t* __restrict__ flags) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    flags[q] = (!elig[q] || overflow[q] || (!positive_only && out_cnt[q] < need)) ? 1 : 0;
}

// signature sort on the device: keys ~sig ascending (= signature descending; the radix sort is stable, so equal
// signatures keep query order), values = query index
__global__ void k_sig_keys(const uint32_t* __restrict__ sig, int32_t nq, uint32_t* __restrict__ key, int32_t* __restrict__ val) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq) { key[i] = ~sig[i]; val[i] = i; }
}
__global__ void k_invert_perm(const int32_t* __restrict__ perm, int32_t nq, int32_t* __restrict__ inv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq) inv[perm[i]] = i;
}

__global__ void k_fill_offsets(int64_t* __restrict__ off, int32_t nq, int64_t stride) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q <= nq) off[q] = (int64_t)q * stride;
}

// all plans again from the current thresholds (after a cross-shard threshold exchange)
__global__ void __launch_bounds__(128) k_replan(const float* __restrict__ thr, int32_t nq, const int32_t* __restrict__ elig,
                                                PlanArgs pa) {
    const int lane = threadIdx.x & 31;
    const int q = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (q >= nq || !elig[q]) return;
    make_plan(pa, q, thr[q], lane);
}

// Cross-shard threshold exchange (doc-sharded callers, br_set_thr_exchange).  After the seeding the shards' thr[Q] are
// gathered and every shard takes the maximum; after a tile launch the shards' current K best fp32 scores of every query
// (the heads of the candidate lists k_tighten has just sorted) are gathered and thr[q] is raised to the K-th largest of the
// world x K values: K distinct docs of the whole corpus score at least that much, so it is a valid lower bound of the
// K-th best score of the WHOLE corpus - the bound a single index would have after the same fraction of its docs - and the
// plans follow.
__global__ void k_xchg_heads(const float* __restrict__ cand_h, const int32_t* __restrict__ cand_cnt, int cap, int32_t nq, int K,
                             float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)nq * K) return;
    const int q = (int)(i / K), j = (int)(i - (int64_t)q * K);
    out[i] = j < min(cand_cnt[q], cap) ? cand_h[(int64_t)q * cap + j] : 0.f;
}
constexpr int XCHG_PER = 16;          // world x K <= 32 x XCHG_PER values per query
__global__ void __launch_bounds__(128) k_xchg_union(const float* __restrict__ gathered, int world, int32_t nq, int n_per,
                                                    int K, float* __restrict__ thr) {
    const int lane = threadIdx.x & 31;
    const int q = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (q >= nq) return;
    const int n = world * n_per;        // n_per = 1: the shards' thresholds (maximum); n_per = K: their K best scores
    float v[XCHG_PER];
#pragma unroll
    for (int j = 0; j < XCHG_PER; ++j) {
        const int i = lane + 32 * j;
        v[j] = -1.f;
        if (i < n) { const int r = i / n_per, c = i - r * n_per; v[j] = gathered[((int64_t)r * nq + q) * n_per + c]; }
    }
    const int rounds = n_per == 1 ? 1 : K;
    float kth = 0.f;
    for (int r = 0; r < rounds; ++r) {
        float m = -1.f;
#pragma unroll
        for (int j = 0; j < XCHG_PER; ++j) m = fmaxf(m, v[j]);
        float M = m;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, o));
        const int winner = __ffs(__ballot_sync(0xffffffffu, m == M)) - 1;
        if (lane == winner) {
            bool removed = false;
#pragma unroll
            for (int j = 0; j < XCHG_PER; ++j)
                if (!removed && v[j] == M) { v[j] = -1.f; removed = true; }
        }
        kth = M;
    }
    if (lane == 0 && kth > thr[q]) thr[q] = kth;
}
static int exchange_thr(br_index* ix, float* thr, int32_t nq, const int32_t* elig, const PlanArgs& pa, cudaStream_t st,
                        const TileArgs* a, float* x_local, float* x_gathered) {
    const int world = ix->thr_exchange_world;
    const int n_per = a ? a->K : 1;
    const float* local = thr;
    if (a) {
        k_xchg_heads<<<blocks_for((int64_t)nq * a->K, 256), 256, 0, st>>>(a->cand_h, a->cand_cnt, a->cap, nq, a->K, x_local);
        BR_CUDA(cudaGetLastError());
        local = x_local;
    }
    const int rc = ix->thr_exchange(local, x_gathered, (int64_t)nq * n_per, (void*)st, ix->thr_exchange_user);
    BR_REQUIRE(rc == 0, BR_ERR_STATE, "br_topk_batch: the threshold exchange callback failed");
    k_xchg_union<<<blocks_for((int64_t)nq * 32, 128), 128, 0, st>>>(x_gathered, world, nq, n_per, a ? a->K : 1, thr);
    BR_CUDA(cudaGetLastError());
    k_replan<<<blocks_for((int64_t)nq * 32, 128), 128, 0, st>>>(thr, nq, elig, pa);
    BR_CUDA(cudaGetLastError());
    ix->stats.kernel_launches += a ? 3 : 2;
    return BR_OK;
}

// The launch schedule of the tile kernel: chunks of growing size, thresholds learnt on the first 2^c units filter the
// next 2^c.  k <= 32: units are whole tiles, and the first chunk holds as many as the candidate buffer certainly takes
// with the thresholds still at their seeds (every sub-range can emit up to ~3k docs before its first tightening).
// Large k: units are sub-ranges - before the first threshold exists everything passes, so the first launch covers only
// as many docs as a candidate region holds (TILE_CAP_BIG / S sub-ranges, half a tile), then grows.
// f(sub_begin, sub_end) is called once per launch, in order; it returns a status (BR_OK to go on).
template <class F>
static int for_each_launch(int n_sub, int k, F&& f) {
    const bool big = k > 32;
    const int unit = big ? 1 : TILE_W;                  // sub-ranges per scheduling unit
    const int n_units = big ? n_sub : (n_sub + TILE_W - 1) / TILE_W;
    int t0 = 0, chunk = big ? std::max(1, TILE_CAP_BIG / TILE_S) : std::max(1, std::min(TILE_CHUNK0, TILE_CAP / (TILE_W * 3 * k)));
    while (t0 < n_units) {
        const int nu = std::min(std::min(chunk, n_units - t0), 32768 * unit);
        BR_TRY(f(t0 * unit, std::min((t0 + nu) * unit, n_sub)));
        t0 += nu;
        chunk *= TILE_GROWTH;
    }
    return BR_OK;
}

template <int QT, bool FILT>
static int launch_tiles(const TileArgs& a0, size_t smem, cudaStream_t st, br_index* ix, int32_t* prev_cnt,
                        int32_t* overflow, const PlanArgs& pa, int exchange_rounds, float* x_local, float* x_gathered) {
    BR_CUDA(cudaFuncSetAttribute(k_tile_score<QT, FILT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));   // per device
    const bool big = a0.cap > TILE_CAP;
    if (big) BR_CUDA(cudaFuncSetAttribute(k_tighten_big, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * TILE_CAP_BIG));
    int round = 0;
    return for_each_launch(a0.n_sub, a0.K, [&](int sub_begin, int sub_end) -> int {
        TileArgs a = a0;
        a.sub_begin = sub_begin;
        a.sub_end = sub_end;
        a.tile0 = a.sub_begin / TILE_W;
        a.tile_end = (a.sub_end + TILE_W - 1) / TILE_W;
        const int ny = a.tile_end - a.tile0;
        // consecutive tiles per CTA: amortises the CTA prologue in the large launches, keeps the small ones wide
        a.tpb = 1;
        while (a.tpb * 2 <= TILE_TPB && ny >= 4 * a.tpb) a.tpb *= 2;
        ix->prof_begin(st);
        k_tile_score<QT, FILT><<<dim3((unsigned)a0.nq, (unsigned)((ny + a.tpb - 1) / a.tpb)), TILE_W * 32, smem, st>>>(a);
        BR_CUDA(cudaGetLastError());
        ix->prof_end(st);
        if (big) k_tighten_big<<<a0.nq, TG_T, 8 * (size_t)a0.cap, st>>>(a0.thr, a0.cand_cnt, prev_cnt, a0.cand, a0.cand_h, a0.K, a0.cap, a0.cap, overflow, pa);
        else k_tighten<<<a0.nq, TGS_T, 0, st>>>(a0.thr, a0.cand_cnt, prev_cnt, a0.cand, a0.cand_h, a0.K, overflow, pa);
        BR_CUDA(cudaGetLastError());
        ix->stats.kernel_launches += 2;
        if (round++ < exchange_rounds) BR_TRY(exchange_thr(ix, a0.thr, a0.nq, a0.elig, pa, st, &a0, x_local, x_gathered));   // same count on every shard
        return BR_OK;
    });
}

int fused_launch_count(const br_index* ix, int32_t k) {
    if (!fused_supported(ix, k, 1)) return 0;
    int n = 0;
    for_each_launch(ix->n_sub, k, [&](int, int) -> int { ++n; return BR_OK; });
    return n;
}

bool fused_supported(const br_index* ix, int32_t k, int32_t nq, bool cos) {
    // 32 < k <= 1024: candidate regions of TILE_CAP_BIG slots per query (16 B each) - bounded to 6 GB of scratch
    const bool k_ok = k <= 32 || (k <= 1024 && (int64_t)nq * TILE_CAP_BIG * 16 <= (6LL << 30));
    return ix->allow_fused && k_ok && (cos || ix->variant != BR_OKAPI_NO_PLUS1) && ix->n_hot > 0 &&
           ix->sub_shift == TILE_SHIFT && ix->skip != nullptr;
}

// Fused path over the whole prepared batch.  h_flags[q] != 0 afterwards -> query q must be served by
// the dense path (not eligible, candidate overflow, or fewer than k docs with a positive score).
// long_pass: the second pass for queries with up to 64 terms / 40 hot terms.
int topk_fused(br_index* ix, const int32_t* q_off, const PrepView& pv, int32_t nq, int32_t k, int dedup,
               int positive_only, int32_t* out_ids, double* out_scores, int32_t* out_counts, cudaStream_t st,
               std::vector<int32_t>* h_flags, bool long_pass, const br_posting* post_table, const DocFilter* filt) {
    // post_table != nullptr: the TF-IDF cosine stage (br_tfidf_cosine_topk) - same kernels over the weight table
    // tf*idf^2/||d|| (all weights >= 0 whatever the idf variant), no deferral (the look-up rows and upper bounds hold
    // BM25 weights), candidates re-scored with Formula::COS
    const bool cos = post_table != nullptr;
    const br_posting* const post = cos ? post_table : ix->post;
    const int n_srows = cos ? 0 : ix->n_srows;
    const int umax = long_pass ? TILE_QT_LONG : TILE_QT;
    const int cap = k <= 32 ? TILE_CAP : TILE_CAP_BIG;
    const int n_tiles = (ix->n_sub + TILE_W - 1) / TILE_W;
    const int64_t n_buckets = (int64_t)n_tiles * nq;
    const int64_t n_scan_blocks = (n_buckets + SCAN_TILE - 1) / SCAN_TILE;
    size_t bytes = 0;
    auto carve = [&](size_t n) { size_t o = bytes; bytes += (n + 255) & ~(size_t)255; return o; };
    const size_t Q = (size_t)nq + 2;
    const size_t o_ent = carve(sizeof(TileEntry) * (size_t)nq * umax), o_ne = carve(4 * (size_t)nq),
                 o_el = carve(4 * Q), o_thr = carve(4 * Q), o_cnt = carve(4 * Q), o_prev = carve(4 * Q), o_ovf = carve(4 * Q),
                 o_dm = carve(4 * Q), o_nu = carve(4 * Q),
                 o_off = carve(8 * Q), o_fl = carve(4 * Q), o_oc = carve(4 * Q), o_ct = carve(16),
                 o_bc = carve(4 * (size_t)(n_buckets + 1)), o_bo = carve(4 * (size_t)(n_buckets + 1)),
                 o_cur = carve(4 * (size_t)(n_buckets + 1)), o_part = carve(4 * (size_t)(n_scan_blocks + 1)),
                 o_poff = carve(8 * (size_t)(n_scan_blocks + 2)),
                 o_cand = carve(4 * (size_t)nq * cap), o_ch = carve(4 * (size_t)nq * cap),
                 o_cs = carve(8 * (size_t)nq * cap), o_perm = carve(4 * Q), o_inv = carve(4 * Q), o_sk = carve(12 * Q),
                 o_xl = carve(4 * Q * (size_t)std::min<int32_t>(k, 32)), o_xg = carve(4 * Q * (size_t)std::min<int32_t>(k, 32) * (size_t)std::max(1, ix->thr_exchange_world));
    BR_TRY(ix->ws_tile.reserve(bytes));
    char* p = ix->ws_tile.as<char>();
    TileEntry* entries = (TileEntry*)(p + o_ent);
    int32_t* n_entries = (int32_t*)(p + o_ne);
    int32_t* elig = (int32_t*)(p + o_el);
    float* thr = (float*)(p + o_thr);
    int32_t* cand_cnt = (int32_t*)(p + o_cnt);
    int32_t* prev_cnt = (int32_t*)(p + o_prev);
    int32_t* overflow = (int32_t*)(p + o_ovf);
    uint32_t* defer_mask = (uint32_t*)(p + o_dm);
    float* ne_ub = (float*)(p + o_nu);
    int64_t* cand_off = (int64_t*)(p + o_off);
    int32_t* flags = (int32_t*)(p + o_fl);
    int32_t* cnt_tmp = out_counts ? out_counts : (int32_t*)(p + o_oc);
    unsigned long long* cold_total = (unsigned long long*)(p + o_ct);
    uint32_t* b_cnt = (uint32_t*)(p + o_bc);
    uint32_t* b_off = (uint32_t*)(p + o_bo);
    uint32_t* b_cur = (uint32_t*)(p + o_cur);
    uint32_t* part = (uint32_t*)(p + o_part);
    int64_t* part_off = (int64_t*)(p + o_poff);
    int32_t* cand = (int32_t*)(p + o_cand);
    float* cand_h = (float*)(p + o_ch);
    double* cand_sc = (double*)(p + o_cs);
    int32_t* perm = (int32_t*)(p + o_perm);
    int32_t* inv_perm = (int32_t*)(p + o_inv);
    float* x_local = (float*)(p + o_xl);
    float* x_gathered = (float*)(p + o_xg);

    // Order the CTAs along grid x by signature (bit 31 = most frequent term): queries that share frequent terms sit next
    // to each other, so CTAs that run at the same time read the same posting slices and look-up rows from L2.  Measured
    // on the C4 workload (B200, 1000 W): the tile kernel takes 48.5 ms per 10k-query step sorted, 49.5 ms in query order.
    {
        uint32_t* key_in = (uint32_t*)(p + o_sk);
        uint32_t* key_out = key_in + Q;
        int32_t* val_in = (int32_t*)(key_out + Q);
        k_sig_keys<<<blocks_for(nq, 256), 256, 0, st>>>(pv.sig, nq, key_in, val_in);
        BR_CUDA(cudaGetLastError());
        size_t tmp_bytes = 0;
        BR_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, key_in, key_out, val_in, perm, nq, 0, 32, st));
        BR_TRY(ix->ws_sort.reserve(tmp_bytes + 16));
        BR_CUDA(cub::DeviceRadixSort::SortPairs(ix->ws_sort.as<void>(), tmp_bytes, key_in, key_out, val_in, perm, nq, 0, 32, st));
        k_invert_perm<<<blocks_for(nq, 256), 256, 0, st>>>(perm, nq, inv_perm);
        BR_CUDA(cudaGetLastError());
        ix->stats.kernel_launches += 2;
    }
    if (ix->ws_cold.cap == 0) BR_TRY(ix->ws_cold.reserve(sizeof(ColdEntry) * std::max<size_t>(1u << 20, (size_t)nq * 2048)));
    for (int attempt = 0; attempt < 2; ++attempt) {
    // one memset covers thr / cand_cnt / prev_cnt / overflow / defer_mask / ne_ub (contiguous carve)
    BR_CUDA(cudaMemsetAsync(p + o_thr, 0, o_off - o_thr, st));
    BR_CUDA(cudaMemsetAsync(cold_total, 0, 16, st));
    k_tile_prep<<<(nq + 3) / 4, 128, 0, st>>>(pv, q_off, ix->hot_slot, ix->row_ptr, nq, umax, entries, n_entries, elig, cold_total,
                                              std::max<int64_t>(1, (ix->n_docs * (int64_t)TILE_DENSE_MIN) >> TILE_SHIFT), perm,
                                              ix->row_slot, n_srows, umax, long_pass ? 64 : 32);
    BR_CUDA(cudaGetLastError());
    k_fill_offsets<<<blocks_for(nq + 1, 256), 256, 0, st>>>(cand_off, nq, cap);
    BR_CUDA(cudaGetLastError());
    ix->stats.kernel_launches += 2;
    // Cold postings -> (tile, query) buckets.  Their number is known on the device only; reading it back here would
    // stall the stream in the middle of the batch, so the scatter writes into the buffer kept from earlier batches
    // (bounded by its capacity) and the total is checked after the batch: a batch that needed more is repeated once
    // with a larger buffer.
    const ColdEntry* cold = nullptr;
    const uint32_t* cold_off = nullptr;
    const uint32_t cold_cap = (uint32_t)std::min<size_t>(ix->ws_cold.cap / sizeof(ColdEntry), 0xffffffffu);
    {
        ColdEntry* d_cold = ix->ws_cold.as<ColdEntry>();
        BR_CUDA(cudaMemsetAsync(b_cnt, 0, 4 * (size_t)(n_buckets + 1), st));
        const unsigned qb = blocks_for((int64_t)nq * 32, 128);
        k_cold_pass<false><<<qb, 128, 0, st>>>(pv, q_off, ix->hot_slot, ix->row_ptr, post, nq, elig, inv_perm, b_cnt, nullptr, 0u);
        BR_CUDA(cudaGetLastError());
        k_scan_reduce<<<(unsigned)n_scan_blocks, SCAN_T, 0, st>>>(b_cnt, n_buckets, part);
        BR_CUDA(cudaGetLastError());
        k_exscan<uint32_t><<<1, 1024, 0, st>>>(part, n_scan_blocks, part_off);
        BR_CUDA(cudaGetLastError());
        k_scan_apply<<<(unsigned)n_scan_blocks, SCAN_T, 0, st>>>(b_cnt, n_buckets, part_off, b_off, b_cur);
        BR_CUDA(cudaGetLastError());
        k_cold_pass<true><<<qb, 128, 0, st>>>(pv, q_off, ix->hot_slot, ix->row_ptr, post, nq, elig, inv_perm, b_cur, d_cold, cold_cap);
        BR_CUDA(cudaGetLastError());
        ix->stats.kernel_launches += 5;
        cold = d_cold;
        cold_off = b_off;
    }
    TileArgs a{post, ix->row_ptr, ix->skip, ix->n_sub, ix->n_docs, entries, n_entries, umax, nq, elig,
               cold_off, cold, cold_cap, ix->dense_rows, ix->n_pad, thr, cand_cnt, cand, cand_h, cap, (int)k, 0, 0, 0, 0, 1, dedup ? 0 : 1, perm, defer_mask, ne_ub, ix->row_slot,
               filt ? filt->bits : nullptr, filt ? filt->words : 0, filt ? filt->row : nullptr};
    const PlanArgs pa{q_off, pv.u_terms, pv.u_mult, pv.u_cnt, ix->ub, ix->row_slot, n_srows, cos ? 0.f : (float)ix->defer_pm * 1e-3f, defer_mask, ne_ub};
    const size_t smem = sizeof(float) * TILE_W * TILE_S + (size_t)umax * (sizeof(TileEntry) + sizeof(int64_t) + sizeof(float) +
                                                                        sizeof(uint32_t) + sizeof(uint2) * TILE_W) +
                        sizeof(NeEntry) * NE_MAX + sizeof(uint16_t) * TILE_W * LIST_CAP + 4 * (6 + TILE_W) + (size_t)TILE_W * umax;
    // threshold exchange with the other shards: only in the regular pass of the first attempt, so that every shard makes
    // exactly 1 + thr_exchange_rounds calls per batch
    const bool exchange = !cos && ix->thr_exchange != nullptr && ix->thr_exchange_rounds >= 0 && !long_pass && attempt == 0 && k <= 32 &&
                          ix->thr_exchange_world * (int)k <= 32 * XCHG_PER;
    const int xr = exchange ? ix->thr_exchange_rounds : 0;
    if (k <= 32) {
        k_seed_thr<<<blocks_for((int64_t)nq * 32, 128), 128, 0, st>>>(post, ix->row_ptr, nq, (int)k, elig, thr, pa,
                                                                      filt ? *filt : DocFilter{});
        BR_CUDA(cudaGetLastError());
        ix->stats.kernel_launches += 1;
    }
    // The thresholds, plans, k_tighten(_big) and the exchange only ever see emitted candidates, which the filtered kernels
    // restrict to allowed docs: they need no filter of their own.
    if (exchange) BR_TRY(exchange_thr(ix, thr, nq, elig, pa, st, nullptr, x_local, x_gathered));
    if (long_pass && filt) BR_TRY((launch_tiles<TILE_QT_LONG, true>(a, smem, st, ix, prev_cnt, overflow, pa, xr, x_local, x_gathered)));
    else if (long_pass) BR_TRY((launch_tiles<TILE_QT_LONG, false>(a, smem, st, ix, prev_cnt, overflow, pa, xr, x_local, x_gathered)));
    else if (filt) BR_TRY((launch_tiles<TILE_QT, true>(a, smem, st, ix, prev_cnt, overflow, pa, xr, x_local, x_gathered)));
    else BR_TRY((launch_tiles<TILE_QT, false>(a, smem, st, ix, prev_cnt, overflow, pa, xr, x_local, x_gathered)));
    BR_TRY(launch_rescore_heads(ix, cos ? Formula::COS : Formula::BM25, q_off, pv, dedup, nq, cap, cand_cnt, cand, cand_sc, st));
    BR_TRY(launch_final_select(cand, cand_sc, cand_off, 0, nq, k, positive_only, out_ids, out_scores, cnt_tmp, st, cand_cnt));
    // with shared thresholds a shard legitimately returns fewer than k docs (the rest of the corpus holds better ones)
    const int32_t need = exchange ? 0 : (int32_t)std::min<int64_t>(k, ix->n_docs);
    k_fused_flags<<<blocks_for(nq, 256), 256, 0, st>>>(elig, overflow, cnt_tmp, nq, need, positive_only, flags);
    BR_CUDA(cudaGetLastError());
    ix->stats.kernel_launches += 3;
    h_flags->resize((size_t)nq);
    unsigned long long h_cold = 0;
    BR_CUDA(cudaMemcpyAsync(h_flags->data(), flags, 4 * (size_t)nq, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaMemcpyAsync(&h_cold, cold_total, sizeof(h_cold), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));                    // the only host synchronisation of the fused path
    BR_REQUIRE(h_cold < (1ull << 32), BR_ERR_UNSUPPORTED, "br_topk_batch: more than 2^32 cold postings in one batch");
    if (h_cold > cold_cap) {                               // the cold buffer was too small: grow it and repeat the batch
        BR_REQUIRE(attempt == 0, BR_ERR_CUDA, "br_topk_batch: cold buffer still too small after growing it");
        BR_TRY(ix->ws_cold.reserve(sizeof(ColdEntry) * (size_t)h_cold + 256));
        continue;
    }
    break;
    }   // attempt
    return BR_OK;
}

}  // namespace br
