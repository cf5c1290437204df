// br_cosine.cu - dense cosine similarity on bf16 embeddings (team_run1.py:269-295):
//   e_hat = e / (||e|| + 1e-10) on both sides, sims = E_hat . q_hat, top-k per query.
//
//   k_row_inv_norm      1/(||x||_2 + 1e-10) per row, fp32                        (HBM-bound, one pass)
//   k_cosine_gemm_qs    brute force, d <= 768: bf16 tcgen05 (UMMA) GEMM on CTA pairs, the pair's block of 224 queries
//                       resident in shared memory while doc tiles stream past it (TMA, 128B swizzle, 3-stage ring);
//                       fp32 accumulators in TMEM; epilogue warps read TMEM with tcgen05.ld, apply
//                       1/(||d||+eps) * 1/(||q||+eps) and keep only scores above the query's running threshold - the
//                       [Q, N] score matrix is never written.  Persistent, warp-specialised
//                       (warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2-9 epilogue).        (tensor-bound)
//   k_cosine_gemm_mc    the same for d > 768 (the query block no longer fits): docs[256-row tile] x queries[256-col
//                       tile] per CTA, the doc tile multicast to a CTA pair
//   k_tighten_cos       between doc chunks of doubling size: threshold := k-th best so far, compact list
//   k_cosine_rerank     per query its own c candidate rows (BM25 top-1000 -> cosine): one warp per
//                       (query, candidate) dot product with 128-bit loads              (gather / HBM-bound)
//   k_cosine_rerank_grouped  per query the rows of its c candidate documents, warps split over rows, best row per
//                       document folded in shared memory                               (gather / HBM-bound)
// This is the only place tensor cores are used: it is the only dense contraction on the path.
#include <cuda.h>
#include <cuda_bf16.h>
#include <math_constants.h>
#include <string.h>

#include "br_common.cuh"
#include "br_kernels.cuh"
#include "br_query.cuh"

namespace br {

constexpr int COS_CAP = 1024;       // candidates kept per query between tighten rounds
constexpr float COS_EPS = 1e-10f;   // team_run1.py:271,276

// ------------------------------------------------------------------------------------------
// row norms
// ------------------------------------------------------------------------------------------
__global__ void k_row_inv_norm(const __nv_bfloat16* __restrict__ x, int64_t n, int32_t d, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (row >= n) return;
    const __nv_bfloat16* p = x + row * d;
    float s = 0.f;
    if ((d & 7) == 0) {
        const uint4* p4 = reinterpret_cast<const uint4*>(p);
        for (int i = lane; i < d / 8; i += 32) {
            const uint4 v = __ldg(p4 + i);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float a = __uint_as_float(w[j] << 16), b = __uint_as_float(w[j] & 0xffff0000u);
                s = fmaf(a, a, s);
                s = fmaf(b, b, s);
            }
        }
    } else {
        for (int i = lane; i < d; i += 32) {
            const float a = __bfloat162float(p[i]);
            s = fmaf(a, a, s);
        }
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[row] = 1.0f / (sqrtf(s) + COS_EPS);
}

// ------------------------------------------------------------------------------------------
// PTX helpers (sm_100a)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
                 "l"(map), "r"(bar), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1,
                                               uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5}], [%2], %3;" ::"r"(dst),
        "l"(map), "r"(bar), "h"(mask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
// 32 lanes x 32 columns of fp32: thread i of the warp gets row (lane quarter base + i), columns [c, c+32)
__device__ __forceinline__ void tc_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte swizzle operand tile (rows of 64 bf16 = 128 B, 8-row swizzle atoms of 1024 B):
// start address >> 4 | SBO (1024 B between 8-row groups) >> 4 at bit 32 | version 1 at bit 46 | layout
// SWIZZLE_128B (2) at bit 61.  LBO is unused for this canonical layout.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3ffffu) >> 4) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// ------------------------------------------------------------------------------------------
// the GEMM + threshold-filter kernel
// ------------------------------------------------------------------------------------------
constexpr int CG_BM = 256, CG_BN = 256, CG_BK = 64, CG_STAGES = 3;   // BM = 2 x 128-row UMMAs sharing the B (query) tile
constexpr int CG_A_BYTES = CG_BM * CG_BK * 2, CG_B_BYTES = CG_BN * CG_BK * 2;
constexpr int CG_STAGE_BYTES = CG_A_BYTES + CG_B_BYTES;
constexpr int CG_THREADS = 320;   // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue of rows 0-127, warps 6-9 of rows 128-255
constexpr size_t CG_SMEM = 1024 /*align slack*/ + (size_t)CG_STAGES * CG_STAGE_BYTES + 2 * CG_BN * sizeof(float) + 256;
// instruction descriptor: D=f32 (1<<4), A=bf16 (1<<7), B=bf16 (1<<10), A,B K-major, N=256 (>>3 at bit 17), M=128 (>>4 at bit 24)
constexpr uint32_t CG_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(CG_BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

struct CosArgs {
    const float* inv_nd;      // [n_docs]
    const float* inv_nq;      // [nq]
    const float* thr;         // [nq] k-th best score so far (-inf initially)
    int32_t* cand_cnt;        // [nq]
    int32_t* cand;            // [nq, COS_CAP] local doc ids
    float* cand_h;            // [nq, COS_CAP]
    int64_t n_docs;
    int32_t nq;
    int32_t d;
    int32_t tile_begin, tile_end;   // doc tiles [tile_begin, tile_end) of CG_BM rows
    int32_t window;                 // query-stationary kernel: doc tiles per L2 window
    DocFilter f;                    // row filter (the <true> instantiations only; last, so the fields above keep their offsets)
};

// The filtered kernels keep each query column's filter row in shared memory behind the barriers (beyond the unfiltered
// layout, so that it stays as it is); a row is tested only where a score has passed the threshold.  doc_allowed's test
// on a row pointer that may be null costs these kernels instructions, so the test stays on frow here.
__device__ __forceinline__ bool cos_row_allowed(const CosArgs& a, int32_t frow, int64_t doc) {
    return frow < 0 || ((__ldg(a.f.bits + (int64_t)frow * a.f.words + (doc >> 5)) >> (doc & 31)) & 1u) != 0u;
}

// Epilogue, query column c of the block (query q): the threshold that acc * inv_d is compared against (thr / inv_q,
// widened so that the rounding of the division keeps a superset), 1 / (||q|| + eps) and, FILT, the column's filter row
template <bool FILT>
__device__ __forceinline__ void cos_stage_column(const CosArgs& a, int q, int c, float* s_thr, float* s_inq, int32_t* s_frow) {
    float th = CUDART_INF_F, iq = 0.f;
    if (q < a.nq) {
        iq = a.inv_nq[q];
        const float raw = __ldcg(a.thr + q) / iq;
        th = raw - fabsf(raw) * 4e-6f;
    }
    s_thr[c] = th;
    s_inq[c] = iq;
    if constexpr (FILT) s_frow[c] = q < a.nq ? a.f.row[q] : -1;
}

// Multicast kernel (d > 768): a CTA computes docs[256-row tile] x queries[256-col tile] with two 128-row UMMAs sharing the
// query tile, fp32 accumulators in 2 x 256 TMEM columns.  CTA pairs share every doc (A) tile - rank r loads rows
// [128r, 128r+128) of it and multicasts them to both CTAs, so the doc operand crosses L2->SM once per pair; each CTA loads
// its own query (B) tile.  Stage release is cluster-wide (both CTAs' UMMAs arrive on both CTAs' empty barriers).
template <bool FILT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CG_THREADS, 1) k_cosine_gemm_mc(const __grid_constant__ CUtensorMap map_docs,
                                                               const __grid_constant__ CUtensorMap map_q, CosArgs a) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;             // 128B swizzle needs 1024-byte alignment
    unsigned char* gen = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t s_tiles = base;
    float* s_thr = reinterpret_cast<float*>(gen + CG_STAGES * CG_STAGE_BYTES);          // [CG_BN] scaled thresholds
    float* s_inq = s_thr + CG_BN;                                                        // [CG_BN] 1/(||q||+eps)
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_inq + CG_BN);                        // full[S] empty[S] tfull[2] tempty[2]
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 12);
    int32_t* s_frow = reinterpret_cast<int32_t*>(bars + 14);                            // [CG_BN] (FILT) filter rows
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };
    auto empty_bar = [&](int s) { return bar0 + 8u * (CG_STAGES + s); };
    auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * CG_STAGES + b); };
    auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * CG_STAGES + 2 + b); };

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_rank();
    const int n_qt = ((a.nq + CG_BN - 1) / CG_BN + 1) / 2;          // query-tile PAIRS
    const int64_t n_tiles = (int64_t)(a.tile_end - a.tile_begin) * n_qt;
    const int64_t t_first = blockIdx.x >> 1, t_step = gridDim.x >> 1;
    const int n_kb = (a.d + CG_BK - 1) / CG_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < CG_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 2); }
        for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                   // peers' barriers are initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int64_t t = t_first; t < n_tiles; t += t_step) {
                const int dt = a.tile_begin + (int)(t / n_qt), qt = 2 * (int)(t % n_qt) + (int)crank;
                for (int kb = 0; kb < n_kb; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    mbar_expect_tx(full_bar(stage), CG_STAGE_BYTES);
                    const uint32_t sa = s_tiles + stage * CG_STAGE_BYTES;
                    tma_load_2d_mc(sa + crank * (CG_A_BYTES / 2), &map_docs, full_bar(stage), kb * CG_BK,
                                   dt * CG_BM + (int)crank * 128, (uint16_t)3);       // my 128 doc rows -> both CTAs
                    tma_load_2d(sa + CG_A_BYTES, &map_q, full_bar(stage), kb * CG_BK, qt * CG_BN);
                    if (++stage == CG_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected lane) =====
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (int64_t t = t_first; t < n_tiles; t += t_step) {
                // both accumulator halves (TMEM columns [0,256) and [256,512)) must have been drained
                mbar_wait(tempty_bar(0), acc_phase ^ 1);
                mbar_wait(tempty_bar(1), acc_phase ^ 1);
                acc_phase ^= 1;
                tc_fence_after();
                for (int kb = 0; kb < n_kb; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint32_t sa = s_tiles + stage * CG_STAGE_BYTES;
                    const uint64_t da0 = umma_desc_sw128(sa), da1 = umma_desc_sw128(sa + CG_A_BYTES / 2);
                    const uint64_t db = umma_desc_sw128(sa + CG_A_BYTES);
#pragma unroll
                    for (int k = 0; k < CG_BK / 16; ++k) {        // UMMA_K = 16 bf16 = 32 bytes: +2 in the >>4 address field
                        tc_mma_bf16(tmem_base, da0 + (uint64_t)(2 * k), db + (uint64_t)(2 * k), CG_IDESC, (kb | k) != 0);
                        tc_mma_bf16(tmem_base + CG_BN, da1 + (uint64_t)(2 * k), db + (uint64_t)(2 * k), CG_IDESC, (kb | k) != 0);
                    }
                    tc_commit_mc(empty_bar(stage), (uint16_t)3);    // slot free in BOTH CTAs once these MMAs retire
                    if (++stage == CG_STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit(tfull_bar(0));                            // accumulators ready for the epilogue warps
                tc_commit(tfull_bar(1));
            }
        }
    } else {
        // ===== epilogue warps: half h = (warp-2)/4 owns doc rows [128h, 128h+128) = TMEM columns [256h, 256h+256);
        //       a warp reads TMEM lanes [32*(warp%4), +32) =====
        const int quarter = warp & 3, half = (warp - 2) >> 2;
        const int et = (int)threadIdx.x - 64;                       // 0..255
        uint32_t acc_phase = 0;
        for (int64_t t = t_first; t < n_tiles; t += t_step) {
            const int dt = a.tile_begin + (int)(t / n_qt), qt = 2 * (int)(t % n_qt) + (int)crank;
            asm volatile("bar.sync 1, 256;" ::: "memory");          // previous tile's thresholds no longer in use
            cos_stage_column<FILT>(a, qt * CG_BN + et, et, s_thr, s_inq, s_frow);
            asm volatile("bar.sync 1, 256;" ::: "memory");          // epilogue warps only
            mbar_wait(tfull_bar(half), acc_phase);
            acc_phase ^= 1;
            tc_fence_after();
            const int64_t doc = (int64_t)dt * CG_BM + half * 128 + quarter * 32 + lane;
            const float inv_d = doc < a.n_docs ? a.inv_nd[doc] : 0.f;
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)half * CG_BN;
            // Common case (nothing passes) is branch-free: m = max_j (acc_j * inv_d - thr_j) over 32 columns with the
            // thresholds read as float4; the next 32 columns are already on their way from TMEM.  Only when m >= 0
            // are the 32 columns rescanned and emitted.
            uint32_t v[2][32];
            tc_ld_32x32(taddr, v[0]);
#pragma unroll
            for (int b = 0; b < (CG_BN / 32); ++b) {
                tc_wait_ld();
                if (b + 1 < CG_BN / 32) tc_ld_32x32(taddr + (b + 1) * 32, v[(b + 1) & 1]);
                const uint32_t (&cur)[32] = v[b & 1];
                const float4* t4 = reinterpret_cast<const float4*>(s_thr + b * 32);
                float m = -CUDART_INF_F;
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 th = t4[j4];
                    m = fmaxf(m, fmaf(__uint_as_float(cur[4 * j4 + 0]), inv_d, -th.x));
                    m = fmaxf(m, fmaf(__uint_as_float(cur[4 * j4 + 1]), inv_d, -th.y));
                    m = fmaxf(m, fmaf(__uint_as_float(cur[4 * j4 + 2]), inv_d, -th.z));
                    m = fmaxf(m, fmaf(__uint_as_float(cur[4 * j4 + 3]), inv_d, -th.w));
                }
                if (m >= 0.f && doc < a.n_docs) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float sc = __uint_as_float(cur[j]) * inv_d;
                        bool pass = sc >= s_thr[b * 32 + j];
                        if constexpr (FILT) pass = pass && cos_row_allowed(a, s_frow[b * 32 + j], doc);
                        if (pass) {
                            const int q = qt * CG_BN + b * 32 + j;
                            const int pos = atomicAdd(a.cand_cnt + q, 1);
                            if (pos < COS_CAP) {
                                a.cand[(int64_t)q * COS_CAP + pos] = (int32_t)doc;
                                a.cand_h[(int64_t)q * COS_CAP + pos] = sc * s_inq[b * 32 + j];
                            }
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(half));
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                   // no CTA exits while its peer can still write into it
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------
// Query-stationary CTA-pair variant (the default for d <= 768): tcgen05.mma.cta_group::2, M = 256 docs per pair
// (128 per CTA = its 128 TMEM lanes), N = 224 queries per pair (112 rows of B in each CTA's shared memory).
//   * the pair's query block stays RESIDENT in shared memory for its whole K extent (12 k-blocks x 14 KB per CTA) while
//     doc tiles stream past it through a 3-stage ring of 16 KB - operand traffic L2->SM drops from 48 KB to 16 KB per
//     64-deep k-block per SM, below what the L2 can deliver at full tensor rate;
//   * the accumulators are double-buffered in TMEM (2 x 224 of the 512 columns), so the epilogue of tile i (tcgen05.ld,
//     normalise, threshold filter) runs under the MMAs of tile i+1;
//   * work units (query block, doc tile) are enumerated query-block-major inside windows of 64 doc tiles (~25 MB
//     of embeddings, L2-resident) and split evenly over the pairs, so a pair reloads its query block only once or
//     twice per window and every doc tile comes from HBM once per launch.
// Barriers live in the leader CTA (rank 0) where the single MMA-issuing thread waits; the peer's TMA loads complete
// on the leader's barriers (.cta_group::2), and tcgen05.commit multicasts the "slot free" / "accumulator ready"
// arrivals to both CTAs.
// ------------------------------------------------------------------------------------------
constexpr int QS_NKB = 12;
constexpr int QS_A_BYTES = 128 * CG_BK * 2;            // 16 KB: this CTA's 128 doc rows of one k-block
constexpr int QS_THREADS = 320;                        // warp 0 TMA, warp 1 MMA / TMEM alloc, warps 2-9 epilogue
// Query block width and doc ring depth: 224 x 3 fills the shared memory; 128 x 8, 160 x 6 and 192 x 5 measured within
// noise of it or slower (DESIGN.md 3.5).
constexpr int QS_BN = 224, QS_STAGES = 3;
constexpr int QS_BNH = QS_BN / 2;                      // query rows held by each CTA
constexpr int QS_B_BYTES = QS_BNH * CG_BK * 2;         // one k-block of them
constexpr size_t QS_SMEM = 1024 + (size_t)QS_NKB * QS_B_BYTES + (size_t)QS_STAGES * QS_A_BYTES + 2 * QS_BN * sizeof(float) + 8 * (2 * QS_STAGES + 6) + 16;
// instruction descriptor: D=f32, A=B=bf16 K-major, N=QS_BN (>>3 at bit 17), M=256 (>>4 at bit 24; the pair's M)
constexpr uint32_t QS_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(QS_BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
constexpr int QS_WINDOW = 64;                          // doc tiles per L2 window (~25 MB of embeddings at d = 768)
static_assert(QS_SMEM <= 232448, "query block + doc ring exceed the shared memory of one SM");
static_assert(QS_BN % 32 == 0 && QS_BN <= 256, "QS_BN: multiple of 32 (epilogue column chunks), two accumulator stages in 512 TMEM columns");

__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {   // shared::cta address -> shared::cluster address in CTA `rank`
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default semantics (release at CTA scope), as CUTLASS ClusterBarrier::arrive does: the consumer only needs the TMEM reads,
    // which tcgen05.wait::ld + tcgen05.fence::before_thread_sync have already ordered; .release.cluster costs a MEMBAR.ALL.GPU
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into MY shared memory whose completion bytes are counted on a barrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
                 "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}

// Work units (query block, doc tile) of one pair.  Doc tiles are taken in windows of `window` tiles (L2-sized); inside a
// window the n_qb x wl units are enumerated query-block-major and split evenly over the pairs, so that ALL pairs work on
// the same window at the same time (its doc rows come from HBM once and from L2 for every other query block) and a
// pair changes its resident query block at most about twice per window.
struct QsIter {
    int n_qb, n_dt, window, pair, n_pairs;
    int w, wl, qb, t;
    int64_t r, re;
    bool valid;
    __device__ __forceinline__ bool open_window() {
        for (; w * window < n_dt; ++w) {
            wl = min(window, n_dt - w * window);
            const int64_t uw = (int64_t)n_qb * wl;
            r = (int64_t)pair * uw / n_pairs;
            re = (int64_t)(pair + 1) * uw / n_pairs;
            if (r < re) {
                qb = (int)(r / wl);
                t = (int)(r - (int64_t)qb * wl);
                return true;
            }
        }
        return false;
    }
    __device__ __forceinline__ QsIter(int n_qb_, int n_dt_, int window_, int pair_, int n_pairs_)
        : n_qb(n_qb_), n_dt(n_dt_), window(window_), pair(pair_), n_pairs(n_pairs_), w(0), wl(0), qb(0), t(0), r(0), re(0) {
        valid = open_window();
    }
    __device__ __forceinline__ int tile() const { return w * window + t; }
    __device__ __forceinline__ void next() {
        if (++r == re) {
            ++w;
            valid = open_window();
        } else if (++t == wl) {
            t = 0;
            ++qb;
        }
    }
};

template <bool FILT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(QS_THREADS, 1) k_cosine_gemm_qs(const __grid_constant__ CUtensorMap map_docs,
                                                               const __grid_constant__ CUtensorMap map_q, CosArgs a) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;             // 128B swizzle needs 1024-byte alignment
    unsigned char* gen = smem_raw + (base - smem_u32(smem_raw));
    const uint32_t s_b = base;                                                // [QS_NKB][112 x 64] resident query block (my half)
    const uint32_t s_a = base + QS_NKB * QS_B_BYTES;                          // [QS_STAGES][128 x 64] doc ring
    float* s_thr = reinterpret_cast<float*>(gen + QS_NKB * QS_B_BYTES + QS_STAGES * QS_A_BYTES);   // [QS_BN]
    float* s_inq = s_thr + QS_BN;                                                                   // [QS_BN]
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_inq + QS_BN);
    uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 2 * QS_STAGES + 6);
    int32_t* s_frow = reinterpret_cast<int32_t*>(bars + 2 * QS_STAGES + 8);             // [QS_BN] (FILT) filter rows
    const uint32_t bar0 = smem_u32(bars);
    auto full_bar = [&](int s) { return bar0 + 8u * s; };                      // leader: doc stage filled (both CTAs' bytes)
    auto empty_bar = [&](int s) { return bar0 + 8u * (QS_STAGES + s); };       // each CTA: doc stage consumed
    const uint32_t bfull_bar = bar0 + 8u * (2 * QS_STAGES);                    // leader: query block resident
    const uint32_t bempty_bar = bar0 + 8u * (2 * QS_STAGES + 1);               // each CTA: query block no longer read
    auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * QS_STAGES + 2 + b); };   // each CTA: accumulator stage ready
    auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * QS_STAGES + 4 + b); };  // leader: accumulator stage drained (16 warps)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t crank = cluster_rank();
    const int n_qb = (a.nq + QS_BN - 1) / QS_BN;
    const int n_dt = a.tile_end - a.tile_begin;
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
    const int n_kb = (a.d + CG_BK - 1) / CG_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < QS_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        mbar_init(bfull_bar, 1);
        mbar_init(bempty_bar, 1);
        for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 16); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                   // the peer's barriers exist before anything arrives on them
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        // ===== TMA producer (both CTAs: my half of the query block, my 128 rows of every doc tile) =====
        if (lane == 0) {
            const uint32_t l_bfull = mapa_rank(bfull_bar, 0);
            int stage = 0, cur_qb = -1;
            uint32_t phase = 0, b_phase = 0;
            for (QsIter it(n_qb, n_dt, a.window, pair, n_pairs); it.valid; it.next()) {
                struct { int qb, tile; } un{it.qb, it.tile()};
                if (un.qb != cur_qb) {
                    cur_qb = un.qb;
                    mbar_wait(bempty_bar, b_phase ^ 1);             // every MMA that read the previous block has retired
                    b_phase ^= 1;
                    if (crank == 0) mbar_expect_tx(bfull_bar, 2u * (uint32_t)n_kb * QS_B_BYTES);
                    for (int kb = 0; kb < n_kb; ++kb)
                        tma_load_2d_pair(s_b + kb * QS_B_BYTES, &map_q, l_bfull, kb * CG_BK, un.qb * QS_BN + (int)crank * QS_BNH);
                }
                const int row0 = (a.tile_begin + un.tile) * CG_BM + (int)crank * 128;
                for (int kb = 0; kb < n_kb; ++kb) {
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    if (crank == 0) mbar_expect_tx(full_bar(stage), 2u * QS_A_BYTES);
                    tma_load_2d_pair(s_a + stage * QS_A_BYTES, &map_docs, mapa_rank(full_bar(stage), 0), kb * CG_BK, row0);
                    if (++stage == QS_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one thread of the leader CTA drives both SMs' tensor cores =====
        if (lane == 0 && crank == 0) {
            int stage = 0, cur_qb = -1, acc = 0;
            uint32_t phase = 0, bf_phase = 0, acc_phase[2] = {0, 0};
            for (QsIter it(n_qb, n_dt, a.window, pair, n_pairs); it.valid; it.next()) {
                struct { int qb, tile; } un{it.qb, it.tile()};
                if (un.qb != cur_qb) {
                    cur_qb = un.qb;
                    mbar_wait(bfull_bar, bf_phase);
                    bf_phase ^= 1;
                }
                mbar_wait(tempty_bar(acc), acc_phase[acc] ^ 1);     // both CTAs' epilogue warps have drained this stage
                acc_phase[acc] ^= 1;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
                for (int kb = 0; kb < n_kb; ++kb) {
                    mbar_wait(full_bar(stage), phase);
                    tc_fence_after();
                    const uint64_t da = umma_desc_sw128(s_a + stage * QS_A_BYTES);
                    const uint64_t db = umma_desc_sw128(s_b + kb * QS_B_BYTES);
#pragma unroll
                    for (int k = 0; k < CG_BK / 16; ++k)
                        tc_mma_bf16_pair(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), QS_IDESC, (kb | k) != 0);
                    tc_commit_pair(empty_bar(stage), (uint16_t)3);   // doc slot free in both CTAs once these MMAs retire
                    if (++stage == QS_STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit_pair(tfull_bar(acc), (uint16_t)3);         // accumulators ready for both CTAs' epilogue warps
                QsIter nx = it;
                nx.next();
                if (!nx.valid || nx.qb != cur_qb) tc_commit_pair(bempty_bar, (uint16_t)3);   // last tile under this query block
                acc ^= 1;
            }
        }
    } else {
        // ===== epilogue warps: warp reads TMEM lanes [32*(warp%4), +32) = doc rows of this CTA's half of the tile; the two
        //       warps of a lane quarter split the query columns.  A tcgen05.ld queues behind the UMMAs already issued, so
        //       ALL of a warp's columns are requested up front (NCH x 16 registers) and waited for once. =====
        constexpr int NCH = QS_BN / 32;                                // 16-column chunks per warp
        const int quarter = warp & 3, chalf = (warp - 2) >> 2;
        const int col0 = chalf * (QS_BN / 2);
        const int et = (int)threadIdx.x - 64;                       // 0..255
        const uint32_t l_tempty0 = mapa_rank(tempty_bar(0), 0), l_tempty1 = mapa_rank(tempty_bar(1), 0);
        int cur_qb = -1, acc = 0;
        uint32_t acc_phase[2] = {0, 0};
        for (QsIter it(n_qb, n_dt, a.window, pair, n_pairs); it.valid; it.next()) {
            struct { int qb, tile; } un{it.qb, it.tile()};
            if (un.qb != cur_qb) {
                cur_qb = un.qb;
                asm volatile("bar.sync 1, 256;" ::: "memory");      // previous block's thresholds no longer in use
                if (et < QS_BN) cos_stage_column<FILT>(a, un.qb * QS_BN + et, et, s_thr, s_inq, s_frow);
                asm volatile("bar.sync 1, 256;" ::: "memory");
            }
            const int64_t doc = (int64_t)(a.tile_begin + un.tile) * CG_BM + (int)crank * 128 + quarter * 32 + lane;
            const float inv_d = doc < a.n_docs ? a.inv_nd[doc] : 0.f;
            mbar_wait(tfull_bar(acc), acc_phase[acc]);
            acc_phase[acc] ^= 1;
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)acc * 256u + (uint32_t)col0;
            // All of the warp's columns are in registers after one wait.  The filter is straight-line code: per chunk
            // the maximum of acc*inv_d - thr, and a predicated copy of the chunk's 16 accumulators when it holds a
            // passing column.  The emission code exists ONCE (ncu on the first version, which emitted from 7 x 16
            // unrolled copies: 35 % of all stall samples were instruction-cache misses on the emission lines).
            // A lane with passing columns in two or more chunks (thresholds still loose) sends its warp through the
            // chunk loop, which reads each chunk again from TMEM; otherwise the accumulator stage goes back to the MMA
            // issuer before anything is emitted.
            uint32_t hv[16];
            int hc = 0, nhc = 0;
            {
                uint32_t v[NCH][16];
#pragma unroll
                for (int c = 0; c < NCH; ++c) tc_ld_32x16(taddr + c * 16, v[c]);
                tc_wait_ld();
#pragma unroll
                for (int j = 0; j < 16; ++j) hv[j] = 0u;
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    const float4* t4 = reinterpret_cast<const float4*>(s_thr + col0 + c * 16);
                    float m = -CUDART_INF_F;
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const float4 th = t4[j4];
                        m = fmaxf(m, fmaf(__uint_as_float(v[c][4 * j4 + 0]), inv_d, -th.x));
                        m = fmaxf(m, fmaf(__uint_as_float(v[c][4 * j4 + 1]), inv_d, -th.y));
                        m = fmaxf(m, fmaf(__uint_as_float(v[c][4 * j4 + 2]), inv_d, -th.z));
                        m = fmaxf(m, fmaf(__uint_as_float(v[c][4 * j4 + 3]), inv_d, -th.w));
                    }
                    const bool hit = doc < a.n_docs && m >= 0.f;
#pragma unroll
                    for (int j = 0; j < 16; ++j) hv[j] = hit ? v[c][j] : hv[j];
                    hc = hit ? c : hc;
                    nhc += hit ? 1 : 0;
                }
            }
            const bool multi = __any_sync(0xffffffffu, nhc > 1);
            if (!multi) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(acc ? l_tempty1 : l_tempty0);
            }
            const int c_begin = multi ? 0 : hc, c_end = multi ? NCH : hc + nhc;
#pragma unroll 1
            for (int c = c_begin; c < c_end; ++c) {
                if (multi) {                                    // warp-uniform
                    tc_ld_32x16(taddr + c * 16, hv);
                    tc_wait_ld();
                }
                if (doc < a.n_docs) {
                    const float* thc = s_thr + col0 + c * 16;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float sc = __uint_as_float(hv[j]) * inv_d;
                        bool pass = sc >= thc[j];
                        if constexpr (FILT) pass = pass && cos_row_allowed(a, s_frow[col0 + c * 16 + j], doc);
                        if (pass) {
                            const int col = col0 + c * 16 + j;
                            const int q = un.qb * QS_BN + col;
                            const int pos = atomicAdd(a.cand_cnt + q, 1);
                            if (pos < COS_CAP) {
                                a.cand[(int64_t)q * COS_CAP + pos] = (int32_t)doc;
                                a.cand_h[(int64_t)q * COS_CAP + pos] = sc * s_inq[col];
                            }
                        }
                    }
                }
            }
            if (multi) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(acc ? l_tempty1 : l_tempty0);
            }
            acc ^= 1;
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                   // no CTA exits (or frees TMEM) while its peer can still touch it
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// bitonic sort of s_h / s_id [0, n_sort) by (score desc, id asc), or, BY_GROUP, of s_h / s_id / s_g by (group asc,
// score desc, id asc); n_sort a power of two
constexpr int TC_T = 256;
template <bool BY_GROUP>
__device__ __forceinline__ void cos_sort(float* s_h, int32_t* s_id, int32_t* s_g, int n_sort) {
    for (int size = 2; size <= n_sort; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int i = threadIdx.x; i < n_sort / 2; i += blockDim.x) {
                const int x = 2 * i - (i & (stride - 1)), y = x + stride;
                const bool up = (x & size) == 0;
                const float hx = s_h[x], hy = s_h[y];
                const int32_t ix = s_id[x], iy = s_id[y];
                bool y_first = hy > hx || (hy == hx && iy < ix);
                if constexpr (BY_GROUP) y_first = s_g[y] < s_g[x] || (s_g[y] == s_g[x] && y_first);
                if (y_first == up) {
                    s_h[x] = hy; s_h[y] = hx; s_id[x] = iy; s_id[y] = ix;
                    if constexpr (BY_GROUP) { const int32_t g = s_g[x]; s_g[x] = s_g[y]; s_g[y] = g; }
                }
            }
        }
    }
    __syncthreads();
}

// threshold := k-th best candidate so far; keep the candidates >= threshold, sorted (score desc, id asc).
// GROUPED (row r in group row_group[r]): the list first keeps one entry per group - its best row, the lowest row on ties
// -, so the threshold is the k-th best DISTINCT-group score so far (only raised) and the kept rows are sorted (score
// desc, row asc) = (score desc, group asc).  Every threshold is the score of k distinct groups, so it never exceeds the
// final k-th best group score and no row of a final top-k group is ever filtered out; rows of a group that is already
// in the list are merged by the next call.
template <bool GROUPED>
__global__ void __launch_bounds__(TC_T) k_tighten_cos(float* __restrict__ thr, int32_t* __restrict__ cand_cnt,
                                                      int32_t* __restrict__ prev_cnt, int32_t* __restrict__ cand,
                                                      float* __restrict__ cand_h, const int32_t* __restrict__ row_group,
                                                      int K, int32_t* __restrict__ overflow) {
    __shared__ float s_h[COS_CAP];
    __shared__ int32_t s_id[COS_CAP];
    __shared__ int s_keep;
    int32_t* s_g = nullptr;
    int* s_nd = nullptr;
    if constexpr (GROUPED) {
        __shared__ int32_t s_g_[COS_CAP];
        __shared__ int s_nd_;
        s_g = s_g_;
        s_nd = &s_nd_;
    }
    const int q = blockIdx.x;
    int n = cand_cnt[q];
    if (n == prev_cnt[q]) return;
    if (n > COS_CAP) {
        if (threadIdx.x == 0) overflow[q] = 1;
        n = COS_CAP;
    }
    int32_t* ids = cand + (int64_t)q * COS_CAP;
    float* hs = cand_h + (int64_t)q * COS_CAP;
    int n_sort = 32;                                   // smallest power of two covering the list
    while (n_sort < n) n_sort <<= 1;
    for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
        const int32_t row = i < n ? ids[i] : 0x7fffffff;
        s_h[i] = i < n ? hs[i] : -CUDART_INF_F;
        s_id[i] = row;
        if constexpr (GROUPED) s_g[i] = i < n ? __ldg(row_group + row) : 0x7fffffff;
    }
    if (threadIdx.x == 0) {
        s_keep = 0;
        if constexpr (GROUPED) *s_nd = 0;
    }
    int nd = n;                                        // distinct entries
    if constexpr (GROUPED) {
        // the first entry of every group run is the group's best row; the others become (-inf, INT_MAX) and sort last
        cos_sort<true>(s_h, s_id, s_g, n_sort);
        nd = 0;                                        // only s_h / s_id change here; s_g is only read
        for (int i = threadIdx.x; i < n_sort; i += blockDim.x) {
            const bool first = i < n && (i == 0 || s_g[i] != s_g[i - 1]);
            nd += first ? 1 : 0;
            if (!first) { s_h[i] = -CUDART_INF_F; s_id[i] = 0x7fffffff; }
        }
        for (int o = 16; o > 0; o >>= 1) nd += __shfl_xor_sync(0xffffffffu, nd, o);
        if ((threadIdx.x & 31) == 0 && nd) atomicAdd(s_nd, nd);
    }
    cos_sort<false>(s_h, s_id, s_g, n_sort);
    if constexpr (GROUPED) nd = *s_nd;
    float th = thr[q];
    if (nd >= K && s_h[K - 1] > th) th = s_h[K - 1];
    int keep = 0;
    for (int i = threadIdx.x; i < nd; i += blockDim.x) keep += (s_h[i] >= th) ? 1 : 0;
    for (int o = 16; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
    if ((threadIdx.x & 31) == 0 && keep) atomicAdd(&s_keep, keep);
    __syncthreads();
    keep = s_keep;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        ids[i] = i < keep ? s_id[i] : -1;
        hs[i] = i < keep ? s_h[i] : 0.f;
    }
    if (threadIdx.x == 0) {
        thr[q] = th;
        cand_cnt[q] = keep;
        prev_cnt[q] = keep;
    }
}

// row_group (may be NULL): the lists hold one row per group, returned as its group id
__global__ void k_cos_output(const int32_t* __restrict__ cand, const float* __restrict__ cand_h,
                             const int32_t* __restrict__ cand_cnt, const int32_t* __restrict__ row_group, int32_t nq,
                             int32_t k, int64_t doc_base, int64_t* __restrict__ out_ids, float* __restrict__ out_sims) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)nq * k) return;
    const int q = (int)(i / k), j = (int)(i - (int64_t)q * k);
    const bool ok = j < cand_cnt[q] && j < COS_CAP;           // lists are sorted by the last k_tighten_cos
    const int32_t row = ok ? cand[(int64_t)q * COS_CAP + j] : 0;
    out_ids[i] = ok ? (int64_t)(row_group ? row_group[row] : row) + doc_base : -1;
    out_sims[i] = ok ? cand_h[(int64_t)q * COS_CAP + j] : 0.f;
}

// ------------------------------------------------------------------------------------------
// grouped (document-level) top-k: row r belongs to group row_group[r], a non-decreasing map, so a group's rows are one
// contiguous run and, between rows of different groups, "row asc" is "group asc".  A group scores the best of its rows.
// ------------------------------------------------------------------------------------------
// Layout check, pass 1: block b looks at rows [b * GC_ROWS, (b + 1) * GC_ROWS): a value outside [0, n_groups) or below
// its predecessor sets info[0]; blk_starts[b] = the rows of the block that start a group run.
constexpr int GC_ROWS = 1024;
__global__ void __launch_bounds__(256) k_group_check(const int32_t* __restrict__ rg, int64_t n_rows, int32_t n_groups,
                                                     int32_t* __restrict__ blk_starts, int32_t* __restrict__ info) {
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    int cnt = 0;
    bool bad = false;
    for (int i = threadIdx.x; i < GC_ROWS; i += blockDim.x) {
        const int64_t r = (int64_t)blockIdx.x * GC_ROWS + i;
        if (r >= n_rows) break;
        const int32_t g = rg[r], p = r > 0 ? rg[r - 1] : -1;
        bad |= g < 0 || g >= n_groups || g < p;
        cnt += g != p ? 1 : 0;
    }
    if (bad) atomicOr(info, 1);
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (threadIdx.x == 0) blk_starts[blockIdx.x] = s_cnt;
}
// Pass 2 (after k_exscan of blk_starts into excl[n_blk + 1]): info[2] = non-empty groups; info[1] = R_k, the shortest
// row prefix holding k distinct groups (the row after the k-th run start), or every row when fewer than k groups are
// non-empty.  Only the block holding the k-th run start does any work.
__global__ void __launch_bounds__(GC_ROWS) k_group_prefix(const int32_t* __restrict__ rg, int64_t n_rows,
                                                          const int64_t* __restrict__ excl, int32_t n_blk, int32_t k,
                                                          int32_t* __restrict__ info) {
    const int64_t total = excl[n_blk];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        info[2] = (int32_t)total;
        if (total < k) info[1] = (int32_t)n_rows;
    }
    if (!(excl[blockIdx.x] < k && k <= excl[blockIdx.x + 1])) return;     // block-uniform
    const int64_t r = (int64_t)blockIdx.x * GC_ROWS + threadIdx.x;
    const bool start = r < n_rows && (r == 0 || rg[r] != rg[r - 1]);
    uint32_t tot;
    const uint32_t ex = block_excl_scan(start ? 1u : 0u, &tot);
    if (start && excl[blockIdx.x] + ex + 1 == k) info[1] = (int32_t)(r + 1);
}

// off[g] = first row of group g (lower bound in the non-decreasing map), g in [0, n_groups]
__global__ void k_group_offsets(const int32_t* __restrict__ rg, int64_t n_rows, int32_t n_groups, int32_t* __restrict__ off) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g > n_groups) return;
    int64_t lo = 0, hi = n_rows;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (rg[mid] < g) lo = mid + 1; else hi = mid;
    }
    off[g] = (int32_t)lo;
}

// A filter over groups -> the same filter over rows: bit r of row f = bit row_group[r] of group row f.  One warp per
// output word.
__global__ void k_group_filter_rows(const uint32_t* __restrict__ gbits, int64_t gwords, int32_t n_frows,
                                    const int32_t* __restrict__ rg, int64_t n_rows, int64_t rwords, uint32_t* __restrict__ rbits) {
    const int lane = threadIdx.x & 31;
    const int64_t n_words = (int64_t)n_frows * rwords;
    for (int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n_words;
         w += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t f = w / rwords, r = (w - f * rwords) * 32 + lane;
        bool on = false;
        if (r < n_rows) {
            const int32_t g = rg[r];
            on = ((__ldg(gbits + f * gwords + (g >> 5)) >> (g & 31)) & 1u) != 0u;
        }
        const uint32_t word = __ballot_sync(0xffffffffu, on);
        if (lane == 0) rbits[w] = word;
    }
}

// Exact pass: per (query, group) the best of the group's row sims ([nr, n_rows], -inf = a row the query may not return)
// -> candidate (group id, score); a group without rows or without an allowed row is an empty slot (-1).
__global__ void k_group_max(const float* __restrict__ sims, int32_t nr, int64_t n_rows, const int32_t* __restrict__ off,
                            int32_t n_groups, int32_t* __restrict__ gid, double* __restrict__ gsc) {
    const int64_t total = (int64_t)nr * n_groups;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / n_groups;
        const int32_t g = (int32_t)(i - r * n_groups);
        const float* s = sims + r * n_rows;
        float m = -CUDART_INF_F;
        for (int32_t row = off[g]; row < off[g + 1]; ++row) m = fmaxf(m, s[row]);
        gid[i] = m > -CUDART_INF_F ? g : -1;
        gsc[i] = (double)m;
    }
}

// ------------------------------------------------------------------------------------------
// candidate re-rank: query q against its own candidate rows
// ------------------------------------------------------------------------------------------
// One lane's share of a row's dot product (s) and squared norm (nn): 2 x 4 bf16 pairs per 16-byte vector, in vector
// order.  Both gather kernels use it, so a row's cosine is the same bits in either.
template <int NV, class QV>   // QV: the lane's query vectors, qv[i] for i < NV (registers, or shared memory)
__device__ __forceinline__ void cos_lane_dot(const uint4 (&dv)[NV], const QV& qv, float& s, float& nn) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const uint32_t wa[4] = {dv[i].x, dv[i].y, dv[i].z, dv[i].w};
        const uint32_t wb[4] = {qv[i].x, qv[i].y, qv[i].z, qv[i].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float a0 = __uint_as_float(wa[e] << 16), a1 = __uint_as_float(wa[e] & 0xffff0000u);
            const float b0 = __uint_as_float(wb[e] << 16), b1 = __uint_as_float(wb[e] & 0xffff0000u);
            s = fmaf(a0, b0, s);
            s = fmaf(a1, b1, s);
            nn = fmaf(a0, a0, nn);
            nn = fmaf(a1, a1, nn);
        }
    }
}

// One CTA per query: each warp keeps the query row in registers (d <= 1024: 4 x 16 B per lane) and walks the
// candidates warp, warp+8, ... four at a time (12-16 independent 128-bit loads in flight per lane).  A candidate id
// outside [-1, n_docs) is never read; it scores -inf and sets *bad (when bad != NULL) in a pass over the list before the
// gather, which leaves the registers of the gather loop as they are (its occupancy bounds the gather rate).
template <int NV>   // 16-byte vectors per lane = ceil(d / 256)
__global__ void __launch_bounds__(256) k_cosine_rerank(const __nv_bfloat16* __restrict__ docs,
                                                       const float* __restrict__ inv_nd, int64_t n_docs, int32_t d,
                                                       const __nv_bfloat16* __restrict__ queries,
                                                       const float* __restrict__ inv_nq, const int32_t* __restrict__ cand,
                                                       int32_t c, float* __restrict__ out, int32_t* __restrict__ bad) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x;
    const int nvec = d / 8;
    const uint4* pq = reinterpret_cast<const uint4*>(queries + (int64_t)q * d);
    uint4 qv[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) qv[i] = lane + 32 * i < nvec ? __ldg(pq + lane + 32 * i) : make_uint4(0, 0, 0, 0);
    const float iq = inv_nq[q];
    const int32_t* cq = cand + (int64_t)q * c;
    if (bad)
        for (int j = threadIdx.x; j < c; j += blockDim.x)
            if (cq[j] < -1 || cq[j] >= n_docs) *bad = 1;
    for (int j0 = warp * 4; j0 < c; j0 += 32) {
        int32_t doc[4];
        uint4 dv[4][NV];
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            doc[x] = j0 + x < c ? cq[j0 + x] : -1;
            const bool ok = doc[x] >= 0 && doc[x] < n_docs;
            const uint4* pd = reinterpret_cast<const uint4*>(docs + (int64_t)(ok ? doc[x] : 0) * d);
#pragma unroll
            for (int i = 0; i < NV; ++i)
                dv[x][i] = ok && lane + 32 * i < nvec ? __ldg(pd + lane + 32 * i) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int x = 0; x < 4; ++x) {
            float s = 0.f, nn = 0.f;
            cos_lane_dot<NV>(dv[x], qv, s, nn);
            for (int o = 16; o > 0; o >>= 1) {
                s += __shfl_xor_sync(0xffffffffu, s, o);
                nn += __shfl_xor_sync(0xffffffffu, nn, o);
            }
            if (lane == 0 && j0 + x < c) {
                const bool ok = doc[x] >= 0 && doc[x] < n_docs;
                const float id = !ok ? 0.f : (inv_nd ? inv_nd[doc[x]] : 1.0f / (sqrtf(nn) + COS_EPS));
                out[(int64_t)q * c + j0 + x] = ok ? s * id * iq : -CUDART_INF_F;
            }
        }
    }
}

__global__ void k_f32_to_f64(const float* __restrict__ in, int64_t n, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}
__global__ void k_rerank_output(const int32_t* __restrict__ ids, const double* __restrict__ sc, int64_t n,
                                float* __restrict__ out_sims) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out_sims[i] = ids[i] >= 0 ? (float)sc[i] : 0.f;
}

// Grouped re-rank: query q against the rows of its candidate GROUPS cand[q, 0..c) (local group ids, -1 = empty slot); a
// group scores the best cosine of its rows.  One CTA per query takes the candidates in chunks of RG_CH: an exclusive
// prefix of their row counts (int64: a list may repeat a large group) flattens the chunk's rows into one range, which
// the warps walk 4 rows at a time (warp w: rows 4w.., stride 32), so the work follows rows, not candidates, and one long
// group keeps every warp busy.  A row finds its candidate by binary search in the prefix; its cosine is computed as
// k_cosine_rerank computes it and folded into the candidate's slot with an atomicMax on order-preserving bits (max is
// exact, so the order of the folds does not matter).  Out: per candidate the group id (-1 for an empty slot, an empty
// group or an id outside [-1, n_groups), which also sets *bad and never addresses off[]) and the best cosine, widened.
constexpr int RG_T = 256, RG_CH = 1024;
// Resident CTAs asked of ptxas, per NV: the gather rate follows the loads in flight per SM.  With the query in shared
// memory this gives 56 / 64 / 80 / 120 registers without spills (4 / 4 / 3 / 2 CTAs, as many as k_cosine_rerank).
#define RG_MIN_BLOCKS(NV) ((NV) <= 2 ? 4 : (NV) == 3 ? 3 : 2)
__device__ __forceinline__ uint32_t f32_order(float x) {     // monotone float -> uint32 (for atomicMax)
    const uint32_t u = __float_as_uint(x);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float f32_unorder(uint32_t e) {
    return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e);
}
struct QStrided {                                            // vector i of a lane's query share in shared memory
    const uint4* p;
    __device__ __forceinline__ uint4 operator[](int i) const { return p[32 * i]; }
};
template <int NV>   // 16-byte vectors per lane = ceil(d / 256)
__global__ void __launch_bounds__(RG_T, RG_MIN_BLOCKS(NV)) k_cosine_rerank_grouped(const __nv_bfloat16* __restrict__ docs,
                                                                const float* __restrict__ inv_nd, int32_t d,
                                                                const int32_t* __restrict__ off, int32_t n_groups,
                                                                const __nv_bfloat16* __restrict__ queries,
                                                                const float* __restrict__ inv_nq, const int32_t* __restrict__ cand,
                                                                int32_t c, int32_t* __restrict__ out_ids,
                                                                double* __restrict__ out_sc, int32_t* __restrict__ bad) {
    constexpr int PER = RG_CH / RG_T;                        // candidates per thread in the prefix pass
    __shared__ int64_t s_pre[RG_CH + 1];                     // exclusive prefix of the row counts; [RG_CH] = chunk total
    __shared__ int32_t s_row0[RG_CH];                        // first row of each candidate's group
    __shared__ uint32_t s_best[RG_CH];                       // f32_order(best cosine so far)
    __shared__ int64_t s_wsum[RG_T / 32];
    __shared__ uint4 s_q[32 * NV];                           // the query row, zero-padded to 32 x NV vectors
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int q = blockIdx.x;
    const int nvec = d / 8;
    const uint4* pq = reinterpret_cast<const uint4*>(queries + (int64_t)q * d);
    for (int i = threadIdx.x; i < 32 * NV; i += RG_T) s_q[i] = i < nvec ? __ldg(pq + i) : make_uint4(0, 0, 0, 0);
    const uint4* qv = s_q + lane;                            // qv[32 i]: read at use, so the query holds no registers
    const float iq = inv_nq[q];
    const int32_t* cq = cand + (int64_t)q * c;
    auto group_of = [&](int j) {                             // validated candidate j of the list, -1 = no rows to read
        const int32_t g = j < c ? cq[j] : -1;
        if (g < -1 || g >= n_groups) { *bad = 1; return -1; }
        return g;
    };
    for (int j0 = 0; j0 < c; j0 += RG_CH) {
        // 1. the chunk's row runs and their prefix
        int64_t cnt[PER], sum = 0;
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            const int jl = threadIdx.x * PER + p;
            const int32_t g = group_of(j0 + jl);
            const int32_t r0 = g >= 0 ? off[g] : 0;
            cnt[p] = g >= 0 ? (int64_t)(off[g + 1] - r0) : 0;
            sum += cnt[p];
            s_row0[jl] = r0;
            s_best[jl] = f32_order(-CUDART_INF_F);
        }
        int64_t incl = sum;
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_wsum[warp] = incl;
        __syncthreads();
        int64_t run = incl - sum;
        for (int w = 0; w < warp; ++w) run += s_wsum[w];
#pragma unroll
        for (int p = 0; p < PER; ++p) {
            s_pre[threadIdx.x * PER + p] = run;
            run += cnt[p];
        }
        if (threadIdx.x == RG_T - 1) s_pre[RG_CH] = run;
        __syncthreads();
        // 2. the rows: 4 in flight per warp, as in k_cosine_rerank
        const int64_t total = s_pre[RG_CH];
        for (int64_t f0 = warp * 4; f0 < total; f0 += 32) {
            // lane x (mod 4) locates row f0 + x: its candidate slot (the last run starting at or before it) and its row
            const int64_t f = f0 + (lane & 3);
            int slot = 0;
#pragma unroll
            for (int step = RG_CH / 2; step > 0; step >>= 1) slot += s_pre[slot + step] <= f ? step : 0;
            const int32_t row = f < total ? s_row0[slot] + (int32_t)(f - s_pre[slot]) : -1;
            uint4 dv[4][NV];
#pragma unroll
            for (int x = 0; x < 4; ++x) {
                const int32_t rx = __shfl_sync(0xffffffffu, row, x);
                const uint4* pd = reinterpret_cast<const uint4*>(docs + (int64_t)(rx >= 0 ? rx : 0) * d);
#pragma unroll
                for (int i = 0; i < NV; ++i)
                    dv[x][i] = rx >= 0 && lane + 32 * i < nvec ? __ldg(pd + lane + 32 * i) : make_uint4(0, 0, 0, 0);
            }
#pragma unroll
            for (int x = 0; x < 4; ++x) {
                float s = 0.f, nn = 0.f;
                cos_lane_dot<NV>(dv[x], QStrided{qv}, s, nn);   // nn is not used: the norms come from inv_nd
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (lane == x && row >= 0) atomicMax(s_best + slot, f32_order(s * inv_nd[row] * iq));
            }
        }
        __syncthreads();
        // 3. one (group, score) per candidate
        for (int jl = threadIdx.x; jl < RG_CH && j0 + jl < c; jl += RG_T) {
            const int64_t i = (int64_t)q * c + j0 + jl;
            const bool has_rows = s_pre[jl + 1] > s_pre[jl];
            out_ids[i] = has_rows ? cq[j0 + jl] : -1;
            out_sc[i] = has_rows ? (double)f32_unorder(s_best[jl]) : 0.0;
        }
        __syncthreads();                                     // the next chunk rewrites the shared arrays
    }
}

// ------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_map(CUtensorMap* m, const void* ptr, int64_t rows, int32_t d, int box_rows) {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        BR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        BR_REQUIRE(p && qres == cudaDriverEntryPointSuccess, BR_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        fn = (PFN_encodeTiled)p;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)d * 2};
    const cuuint32_t box[2] = {(cuuint32_t)CG_BK, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    BR_REQUIRE(r == CUDA_SUCCESS, BR_ERR_CUDA, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
    return BR_OK;
}

int row_inv_norms(const void* emb, int64_t n, int32_t d, float* out, cudaStream_t st) {
    BR_REQUIRE(emb && out && n >= 0 && d > 0, BR_ERR_INVALID, "br_row_inv_norms: bad arguments");
    if (n == 0) return BR_OK;
    k_row_inv_norm<<<blocks_for(n * 32, 256), 256, 0, st>>>((const __nv_bfloat16*)emb, n, d, out);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

// row r of the list: the doc rows [0, n) in order; with a filter (f.row != NULL) -1 (an empty slot of the gather pass)
// for the rows query qs[r] may not return
__global__ void k_iota_rows(int32_t* __restrict__ out, int32_t rows, int64_t n, const int32_t* __restrict__ qs, DocFilter f) {
    const int64_t total = (int64_t)rows * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / n, d = i - r * n;
        out[i] = !f.row || doc_allowed(f.row_of(qs[r]), (uint32_t)d) ? (int32_t)d : -1;
    }
}
__global__ void k_cos_patch(const int32_t* __restrict__ rows, int32_t nr, int32_t k, const int32_t* __restrict__ ids,
                            const float* __restrict__ sims, int64_t doc_base, int64_t* __restrict__ out_ids,
                            float* __restrict__ out_sims) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nr * k) return;
    const int r = i / k, j = i - r * k;
    const int64_t o = (int64_t)rows[r] * k + j;
    out_ids[o] = ids[i] >= 0 ? (int64_t)ids[i] + doc_base : -1;
    out_sims[o] = sims[i];
}

// br_set_cosine_option("kernel", v): 0 auto (query-stationary CTA pairs when d <= 768, else 2-CTA multicast), 1 always
// multicast.  Both kernels return bit-identical results; the switch lets a test pin them against each other.
static int g_cos_kernel = 0;

int set_cosine_option(const char* name, int value) {
    BR_REQUIRE(name, BR_ERR_INVALID, "br_set_cosine_option: null name");
    const std::string n(name);
    if (n == "kernel") { BR_REQUIRE(value >= 0 && value <= 1, BR_ERR_INVALID, "br_set_cosine_option: kernel must be 0 or 1"); g_cos_kernel = value; }
    else { set_error("br_set_cosine_option: unknown option " + n); return BR_ERR_INVALID; }
    return BR_OK;
}

// The launch schedule of the brute-force pass, for the grouped and the ungrouped call: fn(t0, nt) covers doc tiles
// [t0, t0 + nt).  The first `warm_tiles` tiles go in launches of at most `warm_cap` tiles: a query may have no threshold
// there yet, so such a launch can emit every row it covers, and `warm_cap` tiles plus what the list already holds fit its
// COS_CAP slots.  After that the launch size doubles, starting from twice the last warm-up launch.  A launch emits about
// k (growth - 1) candidates per query when a candidate is one row; `grow` < 1 replaces the doubling by launches of
// grow x the tiles covered so far (for groups whose rows pass the threshold together, see cosine_topk).
// Ungrouped: warm_tiles = warm_cap = 1, grow = 1 - one tile, then 2, 4, 8, ...
template <class F>
static int for_each_cos_launch(int n_dt, int warm_tiles, int warm_cap, double grow, F&& fn) {
    int t0 = 0, chunk = 1;
    while (t0 < n_dt) {
        int nt;
        if (t0 < warm_tiles) nt = chunk = std::min(warm_tiles - t0, warm_cap);
        else if (grow >= 1.0) nt = chunk;
        else nt = std::max(1, (int)(t0 * grow));
        nt = std::min(nt, n_dt - t0);
        BR_TRY(fn(t0, nt));
        t0 += nt;
        chunk *= 2;
    }
    return BR_OK;
}

// the gather kernel over explicit candidate rows cand[q, 0..c) -> out[q, c] fp32 cosines (-inf for an empty slot);
// bad (may be NULL) is set when an id is outside [-1, n_docs)
int launch_cos_gather(const void* docs, const float* inv_nd, int64_t n_docs, int32_t d, const void* queries,
                      const float* inv_nq, int32_t nq, const int32_t* cand, int32_t c, float* out, int32_t* bad,
                      cudaStream_t st) {
    BR_REQUIRE(d <= 1024, BR_ERR_UNSUPPORTED, "br_cosine_rerank: embedding dim > 1024");
    const int nv = (d / 8 + 31) / 32;
    auto launch = [&](auto kern) {
        kern<<<nq, 256, 0, st>>>((const __nv_bfloat16*)docs, inv_nd, n_docs, d, (const __nv_bfloat16*)queries, inv_nq, cand, c, out,
                                 bad);
    };
    if (nv <= 1) launch(k_cosine_rerank<1>);
    else if (nv == 2) launch(k_cosine_rerank<2>);
    else if (nv == 3) launch(k_cosine_rerank<3>);
    else launch(k_cosine_rerank<4>);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

// The selection of the re-rank calls: ids / s64 hold nq lists of c (id, float64 score), -1 = an empty slot -> per query
// the top k ids by (score desc, id asc), a repeated id once, with their scores as fp32; -1 / 0.0 pad the rest.
static int select_fixed(const int32_t* ids, const double* s64, int32_t nq, int32_t c, int32_t k, int32_t* out_ids,
                        float* out_sims, cudaStream_t st) {
    StreamScratch tmp(st);
    double* o64;
    BR_TRY(tmp.alloc(&o64, (size_t)nq * k));
    BR_TRY(launch_final_select(ids, s64, nullptr, 0, nq, k, 0, out_ids, o64, nullptr, st, nullptr, c));
    k_rerank_output<<<blocks_for((int64_t)nq * k, 256), 256, 0, st>>>(out_ids, o64, (int64_t)nq * k, out_sims);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

// The layout of a grouped call, checked before anything reads a row through it: a decreasing value or one outside
// [0, n_groups) fails the call `fn`.  Also returns R_k, the shortest row prefix holding k distinct groups (every row when
// fewer than k groups are non-empty), and the number of non-empty groups.
static int check_row_group(const int32_t* row_group, int64_t n_rows, int32_t n_groups, int32_t k, const std::string& fn,
                           cudaStream_t st, int64_t* r_k, int64_t* n_nonempty) {
    const int32_t n_blk = (int32_t)((n_rows + GC_ROWS - 1) / GC_ROWS);
    StreamScratch tmp(st);
    unsigned char* lay;
    BR_TRY(tmp.alloc(&lay, 4 * (size_t)n_blk + 8 * ((size_t)n_blk + 1) + 16));
    int64_t* excl = (int64_t*)lay;
    int32_t* blk = (int32_t*)(excl + n_blk + 1);
    int32_t* info = blk + n_blk;
    BR_CUDA(cudaMemsetAsync(info, 0, 16, st));
    k_group_check<<<n_blk, 256, 0, st>>>(row_group, n_rows, n_groups, blk, info);
    BR_CUDA(cudaGetLastError());
    k_exscan<int32_t><<<1, 1024, 0, st>>>(blk, n_blk, excl);
    BR_CUDA(cudaGetLastError());
    k_group_prefix<<<n_blk, GC_ROWS, 0, st>>>(row_group, n_rows, excl, n_blk, k, info);
    BR_CUDA(cudaGetLastError());
    int32_t h_info[4] = {0, 0, 0, 0};
    BR_CUDA(cudaMemcpyAsync(h_info, info, 16, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!h_info[0], BR_ERR_INVALID, fn + ": row_group must be non-decreasing with values in [0, n_groups)");
    *r_k = h_info[1];
    *n_nonempty = h_info[2];
    return BR_OK;
}

// Grouped call: row r belongs to group row_group[r] (device, non-decreasing, in [0, n_groups)).
struct CosGroups {
    const int32_t* row_group;
    int32_t n_groups;
};

int cosine_topk(const void* docs, const float* inv_nd, int64_t n_docs, int32_t d, const void* queries, int32_t nq,
                int32_t k, int64_t doc_base, int64_t* out_ids, float* out_sims, const br_doc_filter* filter, cudaStream_t st,
                const CosGroups* grp = nullptr) {
    const std::string fn = grp ? "br_cosine_topk_grouped" : "br_cosine_topk";
    BR_REQUIRE(docs && inv_nd && (nq == 0 || (queries && out_ids && out_sims)), BR_ERR_INVALID, fn + ": null pointer");
    BR_REQUIRE(n_docs > 0 && n_docs < (1LL << 31) && nq >= 0, BR_ERR_INVALID, fn + ": bad sizes");
    BR_REQUIRE(d > 0 && d % 8 == 0, BR_ERR_UNSUPPORTED, fn + ": embedding dim must be a multiple of 8 (16-byte rows for TMA)");
    BR_REQUIRE(k >= 1 && k <= 256, BR_ERR_INVALID, fn + ": k must be in [1, 256]");
    BR_REQUIRE(((uintptr_t)docs & 15) == 0 && ((uintptr_t)queries & 15) == 0, BR_ERR_INVALID, fn + ": 16-byte alignment required");
    if (grp) {
        BR_REQUIRE(grp->row_group, BR_ERR_INVALID, fn + ": row_group is null");
        BR_REQUIRE(grp->n_groups >= 1, BR_ERR_INVALID, fn + ": n_groups must be >= 1");
    }
    // a filter is over the ids the call returns: rows, or groups for a grouped call
    BR_TRY(check_doc_filter(filter, grp ? (int64_t)grp->n_groups : n_docs, grp ? "n_groups" : "n_docs", fn));
    if (nq == 0) return BR_OK;
    const int32_t* row_group = grp ? grp->row_group : nullptr;
    const int n_dt = (int)((n_docs + CG_BM - 1) / CG_BM), n_qt = (nq + CG_BN - 1) / CG_BN;
    // Launch schedule.  Ungrouped, the first launch runs without thresholds: every row is a candidate, and one doc tile
    // (CG_BM rows) fits a query's list of COS_CAP.
    static_assert(CG_BM <= COS_CAP, "the first launch must fit the candidate lists");
    int warm_tiles = 1, warm_cap = 1;
    double grow = 1.0;
    if (grp) {
        // One pass over the layout before any GEMM: a decreasing or out-of-range value fails the call, and R_k (the
        // shortest row prefix with k distinct groups) bounds the warm-up.  Until R_k rows are covered a query holds
        // fewer than k groups and no threshold: its list keeps <= k - 1 entries and a launch can emit every row it
        // covers, so warm-up launches cover at most (COS_CAP - (k - 1)) / CG_BM tiles (>= 3).  With singleton groups
        // R_k = k <= CG_BM: one tile, then the ungrouped doubling - the same launches as br_cosine_topk.
        int64_t r_k, n_nonempty;
        BR_TRY(check_row_group(row_group, n_docs, grp->n_groups, k, fn, st, &r_k, &n_nonempty));
        n_nonempty = std::max<int64_t>(n_nonempty, 1);
        warm_tiles = (int)((r_k + CG_BM - 1) / CG_BM);
        warm_cap = (COS_CAP - (k - 1)) / CG_BM;
        // After the warm-up a launch over R new rows passes about k R / S of the groups seen in S rows, and the rows of
        // a passing group tend to pass together (sentences of one document are alike): about k s R / S rows for groups
        // of s rows on average.  Doubling (R = S) keeps that at <= COS_CAP / 4 while k s <= 256 (always, ungrouped);
        // beyond it launches grow by 256 / (k s) of the rows covered so far, so that a launch still fits the lists.
        const double ks = (double)k * (double)n_docs / (double)n_nonempty;
        grow = std::min(1.0, (COS_CAP / 4) / ks);
    }
    static_assert(COS_CAP - 255 >= 3 * CG_BM, "a warm-up launch covers at least 3 tiles for every k <= 256");
    // kernel choice: query-stationary CTA pairs when the query block fits (d <= 768), else 2-CTA multicast
    const bool use_qs = d <= QS_NKB * CG_BK && g_cos_kernel == 0;
    CUtensorMap map_d, map_q;
    BR_TRY(make_map(&map_d, docs, n_docs, d, 128));
    BR_TRY(make_map(&map_q, queries, nq, d, use_qs ? QS_BNH : CG_BN));
    const bool filt = filter != nullptr;
    // the filtered kernels keep the filter rows of their query columns behind the unfiltered layout
    const size_t qs_smem = QS_SMEM + (filt ? sizeof(int32_t) * QS_BN : 0), mc_smem = CG_SMEM + (filt ? sizeof(int32_t) * CG_BN : 0);
    if (filt) {
        BR_CUDA(cudaFuncSetAttribute(k_cosine_gemm_qs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qs_smem));
        BR_CUDA(cudaFuncSetAttribute(k_cosine_gemm_mc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mc_smem));
    } else {
        BR_CUDA(cudaFuncSetAttribute(k_cosine_gemm_qs<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QS_SMEM));   // per device
        BR_CUDA(cudaFuncSetAttribute(k_cosine_gemm_mc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CG_SMEM));
    }
    const size_t Q = (size_t)nq;
    StreamScratch tmp(st);
    float *inv_nq, *thr, *h;
    int32_t *cnt, *prev, *ovf_d, *cand;
    BR_TRY(tmp.alloc(&inv_nq, Q)); BR_TRY(tmp.alloc(&thr, Q)); BR_TRY(tmp.alloc(&cnt, Q)); BR_TRY(tmp.alloc(&prev, Q));
    BR_TRY(tmp.alloc(&ovf_d, Q)); BR_TRY(tmp.alloc(&cand, Q * COS_CAP)); BR_TRY(tmp.alloc(&h, Q * COS_CAP));
    DocFilter fv{};
    int32_t* f_bad = nullptr;
    if (filt) {                                           // [nq] validated rows + the "bad row" flag
        int32_t* frow;
        BR_TRY(tmp.alloc(&frow, Q + 4));
        f_bad = frow + Q;
        BR_CUDA(cudaMemsetAsync(f_bad, 0, 4, st));
        k_filter_rows<<<blocks_for(nq, 256), 256, 0, st>>>(filter->query_row_dev, nq, filter->n_rows, frow, f_bad);
        BR_CUDA(cudaGetLastError());
        fv = DocFilter{filter->bits_dev, filter->words, frow};
    }
    if (filt && grp) {                                    // the group filter as a row filter: the GEMMs test rows
        const int64_t rwords = (n_docs + 31) / 32, n_words = (int64_t)filter->n_rows * rwords;
        uint32_t* rbits;
        BR_TRY(tmp.alloc(&rbits, (size_t)n_words));
        k_group_filter_rows<<<(unsigned)std::min<int64_t>((n_words + 7) / 8, kNumSMs * 64), 256, 0, st>>>(
            filter->bits_dev, filter->words, filter->n_rows, row_group, n_docs, rwords, rbits);
        BR_CUDA(cudaGetLastError());
        fv.bits = rbits;
        fv.words = rwords;
    }
    BR_TRY(row_inv_norms(queries, nq, d, inv_nq, st));
    std::vector<float> ninf(Q, -INFINITY);
    BR_CUDA(cudaMemcpyAsync(thr, ninf.data(), 4 * Q, cudaMemcpyHostToDevice, st));
    BR_CUDA(cudaMemsetAsync(cnt, 0, 4 * Q, st));
    BR_CUDA(cudaMemsetAsync(prev, 0, 4 * Q, st));
    BR_CUDA(cudaMemsetAsync(ovf_d, 0, 4 * Q, st));
    // doc chunks of growing size: thresholds learnt on the docs so far filter the next chunk.  A launch emits about
    // k (growth - 1) candidates per query whatever its size; measured on the config-5 shard an emission costs ~1.7 ns of
    // wall time, which makes doubling (13 launches, ~120 emissions per query) faster than 3x / 4x / 8x growth
    // candidate lists are ~2k long after the first rounds: small CTAs (more of them resident, cheaper barriers)
    constexpr int tighten_t = 64;
    const auto tighten = grp ? k_tighten_cos<true> : k_tighten_cos<false>;
    BR_TRY(for_each_cos_launch(n_dt, warm_tiles, warm_cap, grow, [&](int t0, int nt) {
        CosArgs a{inv_nd, inv_nq, thr, cnt, cand, h, n_docs, nq, d, t0, t0 + nt, QS_WINDOW, fv};
        if (use_qs) {
            const int64_t units = (int64_t)nt * ((nq + QS_BN - 1) / QS_BN);
            const int grid = 2 * (int)std::min<int64_t>(units, kNumSMs / 2);
            if (filt) k_cosine_gemm_qs<true><<<grid, QS_THREADS, qs_smem, st>>>(map_d, map_q, a);
            else k_cosine_gemm_qs<false><<<grid, QS_THREADS, QS_SMEM, st>>>(map_d, map_q, a);
        } else {
            const int grid = 2 * (int)std::min<int64_t>((int64_t)nt * ((n_qt + 1) / 2), kNumSMs / 2);
            if (filt) k_cosine_gemm_mc<true><<<grid, CG_THREADS, mc_smem, st>>>(map_d, map_q, a);
            else k_cosine_gemm_mc<false><<<grid, CG_THREADS, CG_SMEM, st>>>(map_d, map_q, a);
        }
        BR_CUDA(cudaGetLastError());
        tighten<<<nq, tighten_t, 0, st>>>(thr, cnt, prev, cand, h, row_group, k, ovf_d);
        BR_CUDA(cudaGetLastError());
        return BR_OK;
    }));
    k_cos_output<<<blocks_for((int64_t)nq * k, 256), 256, 0, st>>>(cand, h, cnt, row_group, nq, k, doc_base, out_ids, out_sims);
    BR_CUDA(cudaGetLastError());
    std::vector<int32_t> ovf(Q);
    int32_t h_fbad = 0;
    BR_CUDA(cudaMemcpyAsync(ovf.data(), ovf_d, 4 * Q, cudaMemcpyDeviceToHost, st));
    if (f_bad) BR_CUDA(cudaMemcpyAsync(&h_fbad, f_bad, 4, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!h_fbad, BR_ERR_INVALID, fn + ": a filter query_row is outside [-1, n_rows)");
    // A query with more than COS_CAP candidates at or above its threshold in one launch (masses of duplicate / exactly tied
    // embeddings) cannot be served by the filter: those few queries are answered exactly by scoring every doc row with the
    // gather kernel (same normalisation, ties by doc id) - slow (one pass over the embeddings per query) but exact.
    std::vector<int32_t> redo;
    for (int32_t q = 0; q < nq; ++q) if (ovf[(size_t)q]) redo.push_back(q);
    if (redo.empty()) return BR_OK;
    // Any number of such queries: sub-batches of at most 64 bound the scratch (4 B x 64 x n_docs candidate ids).
    // This also covers a corpus whose row order correlates with the queries (every launch then passes far more
    // than COS_CAP rows above the threshold learnt on the rows before it).
    BR_REQUIRE(d <= 1024, BR_ERR_UNSUPPORTED,
               fn + ": candidate overflow (more than 1024 rows at or above a query's running threshold in one "
               "launch) needs the exact gather pass, which supports d <= 1024");
    // Per sub-batch: every row's cosine [nr, n_docs] over the list of all rows (of the allowed rows, filtered), then per
    // (query, id) a float64 score and the re-rank's selection.  The ids are the rows, or for a grouped call the groups
    // [nr, n_groups] with the best of their rows' cosines (a group without rows, or without an allowed row, is an empty
    // slot).
    const int32_t sub = 64;
    const int32_t nr_max = (int32_t)std::min<size_t>(redo.size(), (size_t)sub);
    const int32_t c = grp ? grp->n_groups : (int32_t)n_docs;   // ids per redone query
    char* r_q;
    float *r_inr, *r_s, *r_os;
    int32_t *r_rows, *r_c, *r_id = nullptr, *r_goff, *r_oi;
    double* r_s64;
    BR_TRY(tmp.alloc(&r_q, (size_t)nr_max * d * 2)); BR_TRY(tmp.alloc(&r_inr, (size_t)nr_max)); BR_TRY(tmp.alloc(&r_rows, (size_t)nr_max));
    BR_TRY(tmp.alloc(&r_c, (size_t)nr_max * (size_t)n_docs)); BR_TRY(tmp.alloc(&r_s, (size_t)nr_max * (size_t)n_docs));
    BR_TRY(tmp.alloc(&r_s64, (size_t)nr_max * (size_t)c));
    BR_TRY(tmp.alloc(&r_oi, (size_t)nr_max * k)); BR_TRY(tmp.alloc(&r_os, (size_t)nr_max * k));
    if (grp) {
        BR_TRY(tmp.alloc(&r_id, (size_t)nr_max * (size_t)c)); BR_TRY(tmp.alloc(&r_goff, (size_t)c + 1));
        k_group_offsets<<<blocks_for((int64_t)c + 1, 256), 256, 0, st>>>(row_group, n_docs, c, r_goff);
        BR_CUDA(cudaGetLastError());
    }
    const int32_t* ids = grp ? r_id : r_c;
    for (size_t r0 = 0; r0 < redo.size(); r0 += (size_t)sub) {
        const int32_t nr = (int32_t)std::min<size_t>((size_t)sub, redo.size() - r0);
        for (int32_t i = 0; i < nr; ++i)
            BR_CUDA(cudaMemcpyAsync(r_q + (size_t)i * d * 2, (const char*)queries + (size_t)redo[r0 + (size_t)i] * d * 2,
                                    (size_t)d * 2, cudaMemcpyDeviceToDevice, st));
        BR_CUDA(cudaMemcpyAsync(r_rows, redo.data() + r0, 4 * (size_t)nr, cudaMemcpyHostToDevice, st));
        BR_TRY(row_inv_norms(r_q, nr, d, r_inr, st));
        k_iota_rows<<<kNumSMs * 8, 256, 0, st>>>(r_c, nr, n_docs, r_rows, fv);
        BR_CUDA(cudaGetLastError());
        BR_TRY(launch_cos_gather(docs, inv_nd, n_docs, d, r_q, r_inr, nr, r_c, (int32_t)n_docs, r_s, nullptr, st));
        if (grp)
            k_group_max<<<kNumSMs * 8, 256, 0, st>>>(r_s, nr, n_docs, r_goff, c, r_id, r_s64);
        else
            k_f32_to_f64<<<blocks_for((int64_t)nr * n_docs, 256), 256, 0, st>>>(r_s, (int64_t)nr * n_docs, r_s64);
        BR_CUDA(cudaGetLastError());
        BR_TRY(select_fixed(ids, r_s64, nr, c, k, r_oi, r_os, st));
        k_cos_patch<<<blocks_for((int64_t)nr * k, 256), 256, 0, st>>>(r_rows, nr, k, r_oi, r_os, doc_base, out_ids, out_sims);
        BR_CUDA(cudaGetLastError());
        BR_CUDA(cudaStreamSynchronize(st));               // the next sub-batch rewrites r_q and r_rows
    }
    return BR_OK;
}

int cosine_rerank(const void* docs, const float* inv_nd, int64_t n_docs, int32_t d, const void* queries, int32_t nq,
                  const int32_t* cand, int32_t c, int32_t k, int32_t* out_ids, float* out_sims, cudaStream_t st) {
    BR_REQUIRE(docs && (nq == 0 || (queries && cand && out_ids && out_sims)), BR_ERR_INVALID, "br_cosine_rerank: null pointer");
    BR_REQUIRE(n_docs > 0 && nq >= 0 && c >= 1 && k >= 1 && k <= BR_MAX_K, BR_ERR_INVALID, "br_cosine_rerank: bad sizes");
    BR_REQUIRE(d > 0 && d % 8 == 0, BR_ERR_UNSUPPORTED, "br_cosine_rerank: embedding dim must be a multiple of 8");
    if (nq == 0) return BR_OK;
    const int64_t n_pairs = (int64_t)nq * c;
    StreamScratch tmp(st);
    float *inv_nq, *s;
    double* s64;
    BR_TRY(tmp.alloc(&inv_nq, (size_t)nq + 4)); BR_TRY(tmp.alloc(&s, (size_t)n_pairs)); BR_TRY(tmp.alloc(&s64, (size_t)n_pairs));
    int32_t* bad = (int32_t*)(inv_nq + nq);                // a candidate id outside [-1, n_docs)
    BR_CUDA(cudaMemsetAsync(bad, 0, 4, st));
    BR_TRY(row_inv_norms(queries, nq, d, inv_nq, st));
    BR_TRY(launch_cos_gather(docs, inv_nd, n_docs, d, queries, inv_nq, nq, cand, c, s, bad, st));
    k_f32_to_f64<<<blocks_for(n_pairs, 256), 256, 0, st>>>(s, n_pairs, s64);
    BR_CUDA(cudaGetLastError());
    BR_TRY(select_fixed(cand, s64, nq, c, k, out_ids, out_sims, st));
    int32_t h_bad = 0;
    BR_CUDA(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!h_bad, BR_ERR_INVALID, "br_cosine_rerank: a candidate id is outside [-1, n_docs)");
    return BR_OK;
}

int launch_cos_gather_grouped(const void* docs, const float* inv_nd, int64_t n_rows, int32_t d, const int32_t* row_group,
                              int32_t n_groups, const void* queries, const float* inv_nq, int32_t nq, const int32_t* cand,
                              int32_t c, int32_t* out_ids, double* out_s64, int32_t* bad, const std::string& fn,
                              cudaStream_t st) {
    int64_t r_k, n_nonempty;                               // not used here
    BR_TRY(check_row_group(row_group, n_rows, n_groups, 1, fn, st, &r_k, &n_nonempty));
    StreamScratch tmp(st);
    int32_t* goff;
    BR_TRY(tmp.alloc(&goff, (size_t)n_groups + 1));
    k_group_offsets<<<blocks_for((int64_t)n_groups + 1, 256), 256, 0, st>>>(row_group, n_rows, n_groups, goff);
    BR_CUDA(cudaGetLastError());
    const int nv = (d / 8 + 31) / 32;
    auto launch = [&](auto kern) {
        kern<<<nq, RG_T, 0, st>>>((const __nv_bfloat16*)docs, inv_nd, d, goff, n_groups,
                                  (const __nv_bfloat16*)queries, inv_nq, cand, c, out_ids, out_s64, bad);
    };
    if (nv <= 1) launch(k_cosine_rerank_grouped<1>);
    else if (nv == 2) launch(k_cosine_rerank_grouped<2>);
    else if (nv == 3) launch(k_cosine_rerank_grouped<3>);
    else launch(k_cosine_rerank_grouped<4>);
    BR_CUDA(cudaGetLastError());
    return BR_OK;
}

int cosine_rerank_grouped(const void* docs, const float* inv_nd, int64_t n_rows, int32_t d, const int32_t* row_group,
                          int32_t n_groups, const void* queries, int32_t nq, const int32_t* cand, int32_t c, int32_t k,
                          int32_t* out_ids, float* out_sims, cudaStream_t st) {
    const std::string fn = "br_cosine_rerank_grouped";
    BR_REQUIRE(docs && inv_nd && row_group && (nq == 0 || (queries && cand && out_ids && out_sims)), BR_ERR_INVALID,
               fn + ": null pointer");
    BR_REQUIRE(n_rows > 0 && n_rows < (1LL << 31) && n_groups >= 1 && nq >= 0 && c >= 1 && k >= 1 && k <= BR_MAX_K,
               BR_ERR_INVALID, fn + ": bad sizes");
    BR_REQUIRE(d > 0 && d % 8 == 0, BR_ERR_UNSUPPORTED, fn + ": embedding dim must be a multiple of 8");
    BR_REQUIRE(d <= 1024, BR_ERR_UNSUPPORTED, fn + ": embedding dim > 1024");
    if (nq == 0) return BR_OK;
    // per candidate (group or -1, best cosine), then the same selection as cosine_rerank
    const int64_t n_pairs = (int64_t)nq * c;
    StreamScratch tmp(st);
    float* inv_nq;
    int32_t* ids;
    double* s64;
    BR_TRY(tmp.alloc(&inv_nq, (size_t)nq + 4)); BR_TRY(tmp.alloc(&ids, (size_t)n_pairs)); BR_TRY(tmp.alloc(&s64, (size_t)n_pairs));
    int32_t* bad = (int32_t*)(inv_nq + nq);                // a candidate id outside [-1, n_groups)
    BR_CUDA(cudaMemsetAsync(bad, 0, 4, st));
    BR_TRY(row_inv_norms(queries, nq, d, inv_nq, st));
    BR_TRY(launch_cos_gather_grouped(docs, inv_nd, n_rows, d, row_group, n_groups, queries, inv_nq, nq, cand, c, ids, s64, bad,
                                     fn, st));
    BR_TRY(select_fixed(ids, s64, nq, c, k, out_ids, out_sims, st));
    int32_t h_bad = 0;
    BR_CUDA(cudaMemcpyAsync(&h_bad, bad, 4, cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!h_bad, BR_ERR_INVALID, fn + ": a candidate id is outside [-1, n_groups)");
    return BR_OK;
}

}  // namespace br

extern "C" {

int br_row_inv_norms(const void* emb_bf16_dev, int64_t n, int32_t d, float* out_inv_norm_dev, void* stream) {
    return br::row_inv_norms(emb_bf16_dev, n, d, out_inv_norm_dev, (cudaStream_t)stream);
}

int br_cosine_topk(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_docs, int32_t d,
                   const void* queries_bf16_dev, int32_t nq, int32_t k, int64_t doc_base, int64_t* out_ids_dev,
                   float* out_sims_dev, void* stream) {
    return br::cosine_topk(docs_bf16_dev, doc_inv_norm_dev, n_docs, d, queries_bf16_dev, nq, k, doc_base, out_ids_dev,
                           out_sims_dev, nullptr, (cudaStream_t)stream);
}

int br_cosine_topk_filtered(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_docs, int32_t d,
                            const void* queries_bf16_dev, int32_t nq, int32_t k, int64_t doc_base, int64_t* out_ids_dev,
                            float* out_sims_dev, const br_doc_filter* filter, void* stream) {
    return br::cosine_topk(docs_bf16_dev, doc_inv_norm_dev, n_docs, d, queries_bf16_dev, nq, k, doc_base, out_ids_dev,
                           out_sims_dev, filter, (cudaStream_t)stream);
}

int br_cosine_topk_grouped(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_rows, int32_t d,
                           const int32_t* row_group_dev, int32_t n_groups, const void* queries_bf16_dev, int32_t nq,
                           int32_t k, int64_t doc_base, int64_t* out_ids_dev, float* out_sims_dev,
                           const br_doc_filter* filter, void* stream) {
    const br::CosGroups grp{row_group_dev, n_groups};
    return br::cosine_topk(docs_bf16_dev, doc_inv_norm_dev, n_rows, d, queries_bf16_dev, nq, k, doc_base, out_ids_dev,
                           out_sims_dev, filter, (cudaStream_t)stream, &grp);
}

int br_set_cosine_option(const char* name, int value) { return br::set_cosine_option(name, value); }

int br_cosine_rerank(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_docs, int32_t d,
                     const void* queries_bf16_dev, int32_t nq, const int32_t* cand_ids_dev, int32_t c, int32_t k,
                     int32_t* out_ids_dev, float* out_sims_dev, void* stream) {
    return br::cosine_rerank(docs_bf16_dev, doc_inv_norm_dev, n_docs, d, queries_bf16_dev, nq, cand_ids_dev, c, k, out_ids_dev,
                             out_sims_dev, (cudaStream_t)stream);
}

int br_cosine_rerank_grouped(const void* docs_bf16_dev, const float* doc_inv_norm_dev, int64_t n_rows, int32_t d,
                             const int32_t* row_group_dev, int32_t n_groups, const void* queries_bf16_dev, int32_t nq,
                             const int32_t* cand_groups_dev, int32_t c, int32_t k, int32_t* out_ids_dev,
                             float* out_sims_dev, void* stream) {
    return br::cosine_rerank_grouped(docs_bf16_dev, doc_inv_norm_dev, n_rows, d, row_group_dev, n_groups, queries_bf16_dev, nq,
                                     cand_groups_dev, c, k, out_ids_dev, out_sims_dev, (cudaStream_t)stream);
}

}  // extern "C"
