// br_hybrid.cu - hybrid retrieval: one ranking from a BM25 candidate list B and a dense cosine candidate list D per query.
//
//   k_fuse_union       per query: validate the ids, build the id-sorted distinct union of B and D; for RRF also the
//                      fused score of every member from its first-occurrence ranks
//   k_fuse_linear      per query: min / max of the members' exact BM25 and cosine over the union, normalised scores and
//                      their convex combination
//   k_fuse_components  the two components of every returned doc, looked up in the id-sorted union
//
// The linear mode's components are not recomputed here: the BM25 of a member is k_rescore_heads over the union (the
// float64 re-score br_topk_batch ranks by), its cosine the gather kernel of br_cosine_rerank (flat) or of
// br_cosine_rerank_grouped (grouped).  Selection is k_final_select in its fixed-stride form.  Every float64 operation
// of the fusion is an explicit __d*_rn intrinsic, so no FMA contraction can make it differ from a numpy restatement.
#include <math_constants.h>

#include <cmath>

#include "br_common.cuh"
#include "br_kernels.cuh"
#include "br_query.cuh"

namespace br {

constexpr int FU_T = 256, FU_N = 2 * BR_MAX_K;   // nb + nd <= FU_N: a union is one k_final_select pass (its FS_N keys)
constexpr uint64_t FU_NONE = ~0ull;

// One CTA per query.  Slot j of list L (0 = B, 1 = D) with a valid id becomes the key id << 11 | L << 10 | j, so the
// ascending sort puts each id's entries together, its B entries first, each list in slot order: an id's first entry is
// its member head, and its first D entry is the first entry with L = 1 of the run.  Out: u_ids[q, 0..W) the members in
// id order, -1 padded; u_cnt[q] their number; rrf: u_f[q, m] = w_b / (c + r_b) + w_d / (c + r_d), a term omitted when
// the member is not in that list.  An id outside [-1, n_ids) sets *bad and is dropped, never used.
__global__ void __launch_bounds__(FU_T) k_fuse_union(const int32_t* __restrict__ B, int32_t nb, const int32_t* __restrict__ D,
                                                     int32_t nd, int64_t n_ids, int rrf, double rrf_c, double w_b, double w_d,
                                                     int32_t* __restrict__ u_ids, int32_t* __restrict__ u_cnt,
                                                     double* __restrict__ u_f, int32_t* __restrict__ bad) {
    __shared__ uint64_t keys[FU_N];
    __shared__ int32_t s_rb[FU_N], s_rd[FU_N];             // per member: rank in B / D (0: absent)
    const int q = blockIdx.x;
    const int W = nb + nd;
    int n_sort = 2;
    while (n_sort < W) n_sort <<= 1;
    for (int i = threadIdx.x; i < n_sort; i += FU_T) {
        uint64_t key = FU_NONE;
        if (i < W) {
            const int list = i >= nb ? 1 : 0, slot = list ? i - nb : i;
            const int32_t id = list ? D[(int64_t)q * nd + slot] : B[(int64_t)q * nb + slot];
            if (id < -1 || id >= n_ids) *bad = 1;
            else if (id >= 0) key = (uint64_t)id << 11 | (uint64_t)list << 10 | (uint64_t)slot;
        }
        keys[i] = key;
    }
    for (int size = 2; size <= n_sort; size <<= 1) {       // bitonic, ascending
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < n_sort / 2; i += FU_T) {
                const int a = 2 * i - (i & (stride - 1)), b = a + stride;
                const bool up = (a & size) == 0;
                const uint64_t ka = keys[a], kb = keys[b];
                if ((kb < ka) == up) { keys[a] = kb; keys[b] = ka; }
            }
        }
    }
    __syncthreads();
    // member index of every entry: inclusive count of run heads (FU_N / FU_T entries per thread, blocked)
    constexpr int PER = FU_N / FU_T;
    auto key_at = [&](int i) { return i < n_sort ? keys[i] : FU_NONE; };
    uint32_t head[PER], sum = 0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int i = threadIdx.x * PER + j;
        const uint64_t k = key_at(i);
        head[j] = k != FU_NONE && (i == 0 || (k >> 11) != (key_at(i - 1) >> 11)) ? 1u : 0u;
        sum += head[j];
    }
    uint32_t total;
    const uint32_t ex = block_excl_scan(sum, &total);
    uint32_t m = ex;                                       // heads before this thread's entry j, then its member index + 1
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        m += head[j];
        if (!head[j]) continue;
        const uint64_t k = key_at(threadIdx.x * PER + j);
        const int r = (int)(k & 1023) + 1;
        const bool in_d = (k >> 10) & 1;
        u_ids[(int64_t)q * W + m - 1] = (int32_t)(k >> 11);
        s_rb[m - 1] = in_d ? 0 : r;
        s_rd[m - 1] = in_d ? r : 0;
    }
    __syncthreads();
    m = ex;
#pragma unroll
    for (int j = 0; j < PER; ++j) {                        // the first D entry of a run that starts with B entries
        const int i = threadIdx.x * PER + j;
        m += head[j];
        const uint64_t k = key_at(i);
        if (!head[j] && k != FU_NONE && ((k >> 10) & 1) && !((key_at(i - 1) >> 10) & 1)) s_rd[m - 1] = (int)(k & 1023) + 1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < W; i += FU_T) {
        const int64_t o = (int64_t)q * W + i;
        if (i >= (int)total) u_ids[o] = -1;
        if (!rrf) continue;
        double f = 0.0;
        if (i < (int)total) {
            const int rb = s_rb[i], rd = s_rd[i];
            const double tb = rb ? __ddiv_rn(w_b, __dadd_rn(rrf_c, (double)rb)) : 0.0;
            const double td = rd ? __ddiv_rn(w_d, __dadd_rn(rrf_c, (double)rd)) : 0.0;
            f = rb && rd ? __dadd_rn(tb, td) : rb ? tb : td;
        }
        u_f[o] = f;
    }
    if (threadIdx.x == 0) u_cnt[q] = (int32_t)total;
}

// block-wide min and max of (b, c) over FL_T threads; every thread gets the result
constexpr int FL_T = 256;
__device__ __forceinline__ void block_minmax(double (&v)[4]) {   // {min_b, max_b, min_c, max_c}
    __shared__ double s_v[4][FL_T / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v[0] = fmin(v[0], __shfl_xor_sync(0xffffffffu, v[0], o));
        v[1] = fmax(v[1], __shfl_xor_sync(0xffffffffu, v[1], o));
        v[2] = fmin(v[2], __shfl_xor_sync(0xffffffffu, v[2], o));
        v[3] = fmax(v[3], __shfl_xor_sync(0xffffffffu, v[3], o));
    }
    if (lane == 0)
        for (int j = 0; j < 4; ++j) s_v[j][warp] = v[j];
    __syncthreads();
    for (int w = 0; w < FL_T / 32; ++w) {
        v[0] = fmin(v[0], s_v[0][w]);
        v[1] = fmax(v[1], s_v[1][w]);
        v[2] = fmin(v[2], s_v[2][w]);
        v[3] = fmax(v[3], s_v[3][w]);
    }
}

// (s - lo) / (hi - lo), 0 when hi == lo
__device__ __forceinline__ double minmax_norm(double s, double lo, double hi) {
    return hi == lo ? 0.0 : __ddiv_rn(__dsub_rn(s, lo), __dsub_rn(hi, lo));
}

// One CTA per query over its u_cnt[q] members (stride W): s_b the exact BM25, the cosine from cos_f (flat: every member
// is a row) or from g_ids / g_s64 (grouped: g_ids < 0 = no rows).  Out: f = alpha n_b + (1 - alpha) n_c and the member's
// cosine as fp32, NaN without rows (in place of cos_f when flat).
__global__ void __launch_bounds__(FL_T) k_fuse_linear(const int32_t* __restrict__ u_cnt, int32_t W,
                                                      const double* __restrict__ s_b, const float* cos_f,
                                                      const int32_t* __restrict__ g_ids, const double* __restrict__ g_s64,
                                                      double alpha, double* __restrict__ f, float* cos_out) {
    const int q = blockIdx.x;
    const int n = u_cnt[q];
    const int64_t base = (int64_t)q * W;
    double v[4] = {CUDART_INF, -CUDART_INF, CUDART_INF, -CUDART_INF};
    for (int i = threadIdx.x; i < n; i += FL_T) {
        const double b = s_b[base + i];
        v[0] = fmin(v[0], b);
        v[1] = fmax(v[1], b);
        if (!g_ids || g_ids[base + i] >= 0) {
            const double c = g_ids ? g_s64[base + i] : (double)cos_f[base + i];
            v[2] = fmin(v[2], c);
            v[3] = fmax(v[3], c);
        }
    }
    block_minmax(v);
    const double one_m_alpha = __dsub_rn(1.0, alpha);
    for (int i = threadIdx.x; i < n; i += FL_T) {
        const bool has = !g_ids || g_ids[base + i] >= 0;
        const float c = g_ids ? (float)g_s64[base + i] : cos_f[base + i];
        const double nb = minmax_norm(s_b[base + i], v[0], v[1]);
        const double nc = has ? minmax_norm((double)c, v[2], v[3]) : 0.0;
        f[base + i] = __dadd_rn(__dmul_rn(alpha, nb), __dmul_rn(one_m_alpha, nc));
        cos_out[base + i] = has ? c : CUDART_NAN_F;
    }
}

// out_bm25 / out_cos (either may be NULL) of the selected ids: the member's entry in the id-sorted union; 0 pads
__global__ void k_fuse_components(const int32_t* __restrict__ sel, int32_t nq, int32_t k, const int32_t* __restrict__ u_ids,
                                  const int32_t* __restrict__ u_cnt, int32_t W, const double* __restrict__ s_b,
                                  const float* __restrict__ s_c, double* __restrict__ out_bm25, float* __restrict__ out_cos) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)nq * k) return;
    const int32_t q = (int32_t)(i / k), id = sel[i];
    const int32_t* u = u_ids + (int64_t)q * W;
    int lo = 0, hi = u_cnt[q];
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (u[mid] < id) lo = mid + 1; else hi = mid;
    }
    const bool ok = id >= 0;
    if (out_bm25) out_bm25[i] = ok ? s_b[(int64_t)q * W + lo] : 0.0;
    if (out_cos) out_cos[i] = ok ? s_c[(int64_t)q * W + lo] : 0.f;
}

// ------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------
// The checks both calls share: list widths, k, and the pointers a non-empty batch reads or writes.
static int check_lists(const int32_t* B, int32_t nb, const int32_t* D, int32_t nd, int32_t nq, int32_t k,
                       const int32_t* out_ids, const double* out_scores, const std::string& fn) {
    BR_REQUIRE(nq >= 0 && nb >= 0 && nd >= 0 && nb <= BR_MAX_K && nd <= BR_MAX_K && nb + nd >= 1, BR_ERR_INVALID,
               fn + ": nb and nd must be in [0, BR_MAX_K] with nb + nd >= 1");
    BR_REQUIRE(k >= 1 && k <= BR_MAX_K, BR_ERR_INVALID, fn + ": k must be in [1, BR_MAX_K]");
    BR_REQUIRE(nq == 0 || ((B || nb == 0) && (D || nd == 0) && out_ids && out_scores), BR_ERR_INVALID, fn + ": null pointer");
    return BR_OK;
}

static int report_bad(const int32_t* bad, const int32_t* prep_bad, const std::string& fn, const char* ids, cudaStream_t st) {
    int32_t h_bad[2] = {0, 0};
    BR_CUDA(cudaMemcpyAsync(h_bad, bad, 4, cudaMemcpyDeviceToHost, st));
    if (prep_bad) BR_CUDA(cudaMemcpyAsync(h_bad + 1, prep_bad, 4, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!h_bad[0], BR_ERR_INVALID, fn + ": a candidate id is outside [-1, " + ids + ")");
    BR_REQUIRE(!h_bad[1], BR_ERR_INVALID, fn + ": q_offsets run past n_terms");
    return BR_OK;
}

int fuse_rrf(const int32_t* B, int32_t nb, const int32_t* D, int32_t nd, int64_t n_docs, int32_t nq, double rrf_c,
             double w_b, double w_d, int32_t k, int32_t* out_ids, double* out_scores, int32_t* out_counts, cudaStream_t st) {
    const std::string fn = "br_fuse_rrf";
    BR_TRY(check_lists(B, nb, D, nd, nq, k, out_ids, out_scores, fn));
    BR_REQUIRE(n_docs >= 0 && n_docs <= INT32_MAX, BR_ERR_INVALID, fn + ": n_docs must be in [0, 2^31)");
    BR_REQUIRE(std::isfinite(rrf_c) && rrf_c >= 0.0, BR_ERR_INVALID, fn + ": rrf_c must be finite and >= 0");
    BR_REQUIRE(std::isfinite(w_b) && std::isfinite(w_d) && w_b >= 0.0 && w_d >= 0.0 && (w_b > 0.0 || w_d > 0.0),
               BR_ERR_INVALID, fn + ": weights must be finite, >= 0 and not both 0");
    if (nq == 0) return BR_OK;
    const int32_t W = nb + nd;
    const size_t n = (size_t)nq * W;
    StreamScratch tmp(st);
    int32_t *u_ids, *u_cnt;
    double* f;
    BR_TRY(tmp.alloc(&u_ids, n)); BR_TRY(tmp.alloc(&f, n)); BR_TRY(tmp.alloc(&u_cnt, (size_t)nq + 4));
    int32_t* bad = u_cnt + nq;
    BR_CUDA(cudaMemsetAsync(bad, 0, 4, st));
    k_fuse_union<<<nq, FU_T, 0, st>>>(B, nb, D, nd, n_docs, 1, rrf_c, w_b, w_d, u_ids, u_cnt, f, bad);
    BR_CUDA(cudaGetLastError());
    BR_TRY(launch_final_select(u_ids, f, nullptr, 0, nq, k, 0, out_ids, out_scores, out_counts, st, u_cnt, W));
    return report_bad(bad, nullptr, fn, "n_docs", st);
}

int fuse_linear(br_index* ix, const int32_t* q_terms, const int32_t* q_off, int32_t nq, int32_t n_terms, int dedup,
                const void* docs, const float* inv_nd, int64_t n_rows, int32_t d, const int32_t* row_group, const void* queries,
                const int32_t* B, int32_t nb, const int32_t* D, int32_t nd, double alpha, int32_t k, int32_t* out_ids,
                double* out_scores, double* out_bm25, float* out_cos, int32_t* out_counts, cudaStream_t st) {
    const std::string fn = "br_fuse_linear";
    BR_TRY(check_lists(B, nb, D, nd, nq, k, out_ids, out_scores, fn));
    BR_REQUIRE(ix && docs && inv_nd && (nq == 0 || (q_terms && q_off && queries)), BR_ERR_INVALID, fn + ": null pointer");
    BR_REQUIRE(ix->finalized, BR_ERR_STATE, fn + ": call br_index_finalize first");
    BR_REQUIRE(alpha >= 0.0 && alpha <= 1.0, BR_ERR_INVALID, fn + ": alpha must be in [0, 1]");
    BR_REQUIRE(d > 0 && d % 8 == 0, BR_ERR_UNSUPPORTED, fn + ": embedding dim must be a multiple of 8");
    BR_REQUIRE(d <= 1024, BR_ERR_UNSUPPORTED, fn + ": embedding dim > 1024");
    if (row_group) BR_REQUIRE(n_rows > 0 && n_rows < (1LL << 31), BR_ERR_INVALID, fn + ": n_rows must be in [1, 2^31)");
    else BR_REQUIRE(n_rows == ix->n_docs, BR_ERR_INVALID, fn + ": without row_group, n_rows must equal the index's n_docs");
    if (nq == 0) return BR_OK;
    BR_CUDA(cudaSetDevice(ix->device));
    const int32_t W = nb + nd;
    const size_t n = (size_t)nq * W;
    StreamScratch tmp(st);
    int32_t *u_ids, *u_cnt;
    double *f, *s_b;
    float* s_c;
    BR_TRY(tmp.alloc(&u_ids, n)); BR_TRY(tmp.alloc(&f, n)); BR_TRY(tmp.alloc(&s_b, n)); BR_TRY(tmp.alloc(&s_c, n));
    BR_TRY(tmp.alloc(&u_cnt, 2 * (size_t)nq + 4));
    float* inv_nq = (float*)(u_cnt + nq);
    int32_t* bad = u_cnt + 2 * nq;
    BR_CUDA(cudaMemsetAsync(bad, 0, 4, st));
    k_fuse_union<<<nq, FU_T, 0, st>>>(B, nb, D, nd, ix->n_docs, 0, 0.0, 0.0, 0.0, u_ids, u_cnt, nullptr, bad);
    BR_CUDA(cudaGetLastError());
    // BM25: br_topk_batch's query preparation and float64 re-score over the union
    PrepView pv;
    int64_t* chunk_start;
    BR_TRY(prep_queries(ix, q_terms, q_off, nq, dedup, st, &pv, &chunk_start, n_terms));
    BR_TRY(launch_rescore_heads(ix, Formula::BM25, q_off, pv, dedup, nq, W, u_cnt, u_ids, s_b, st));
    // cosine: the re-rank gather over the union
    BR_TRY(row_inv_norms(queries, nq, d, inv_nq, st));
    const int32_t* g_ids = nullptr;
    const double* g_s64 = nullptr;
    if (row_group) {
        int32_t* gid;
        double* g64;
        BR_TRY(tmp.alloc(&gid, n)); BR_TRY(tmp.alloc(&g64, n));
        BR_TRY(launch_cos_gather_grouped(docs, inv_nd, n_rows, d, row_group, (int32_t)ix->n_docs, queries, inv_nq, nq, u_ids, W,
                                         gid, g64, bad, fn, st));
        g_ids = gid;
        g_s64 = g64;
    } else {
        BR_TRY(launch_cos_gather(docs, inv_nd, n_rows, d, queries, inv_nq, nq, u_ids, W, s_c, nullptr, st));
    }
    k_fuse_linear<<<nq, FL_T, 0, st>>>(u_cnt, W, s_b, s_c, g_ids, g_s64, alpha, f, s_c);
    BR_CUDA(cudaGetLastError());
    BR_TRY(launch_final_select(u_ids, f, nullptr, 0, nq, k, 0, out_ids, out_scores, out_counts, st, u_cnt, W));
    if (out_bm25 || out_cos) {
        k_fuse_components<<<blocks_for((int64_t)nq * k, 256), 256, 0, st>>>(out_ids, nq, k, u_ids, u_cnt, W, s_b, s_c, out_bm25,
                                                                            out_cos);
        BR_CUDA(cudaGetLastError());
    }
    return report_bad(bad, pv.bad, fn, "n_docs", st);
}

}  // namespace br

extern "C" {

int br_fuse_rrf(const int32_t* bm25_ids_dev, int32_t nb, const int32_t* dense_ids_dev, int32_t nd, int64_t n_docs,
                int32_t nq, double rrf_c, double w_bm25, double w_dense, int32_t k, int32_t* out_ids_dev,
                double* out_scores_dev, int32_t* out_counts_dev, void* stream) {
    return br::fuse_rrf(bm25_ids_dev, nb, dense_ids_dev, nd, n_docs, nq, rrf_c, w_bm25, w_dense, k, out_ids_dev, out_scores_dev,
                        out_counts_dev, (cudaStream_t)stream);
}

int br_fuse_linear(br_index* ix, const int32_t* q_terms_dev, const int32_t* q_offsets_dev, int32_t nq, int32_t n_terms,
                   int dedup, const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_rows, int32_t d,
                   const int32_t* row_group_dev, const void* queries_bf16_dev, const int32_t* bm25_ids_dev, int32_t nb,
                   const int32_t* dense_ids_dev, int32_t nd, double alpha, int32_t k, int32_t* out_ids_dev,
                   double* out_scores_dev, double* out_bm25_dev, float* out_cos_dev, int32_t* out_counts_dev, void* stream) {
    return br::fuse_linear(ix, q_terms_dev, q_offsets_dev, nq, n_terms, dedup, docs_bf16_dev, doc_inv_norm_dev, n_rows, d,
                           row_group_dev, queries_bf16_dev, bm25_ids_dev, nb, dense_ids_dev, nd, alpha, k, out_ids_dev,
                           out_scores_dev, out_bm25_dev, out_cos_dev, out_counts_dev, (cudaStream_t)stream);
}

}  // extern "C"
