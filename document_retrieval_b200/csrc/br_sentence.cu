// br_sentence.cu - sentence -> document post-processing of the sentence-level retrieval (implementation 3 of the
// reference): walk a query's ranked sentences, keep the first occurrence of every parent doc, stop at k docs
// (team_run1.py:286-294).
#include "br_common.cuh"
#include "br_kernels.cuh"

namespace br {

// One warp per query.  The docs kept so far live one per lane (k <= 32); every chunk of 32 ranked sentences is mapped
// to docs, compared with the kept ones (shuffles) and within the chunk (the first lane of each __match_any group
// wins), and the survivors are appended in rank order.
__global__ void __launch_bounds__(128) k_dedupe_first_docs(const int64_t* __restrict__ sent, const int32_t* __restrict__ s2d,
                                                           int64_t n_sent, int32_t nq, int32_t n, int32_t k,
                                                           int64_t* __restrict__ out, int* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int q = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (q >= nq) return;
    const int64_t* row = sent + (int64_t)q * n;
    int64_t* orow = out + (int64_t)q * k;
    int32_t kept = -2;                  // lane j: j-th kept doc (-2: none yet)
    int cnt = 0;
    for (int base = 0; base < n && cnt < k; base += 32) {
        const int i = base + lane;
        const int64_t sid = i < n ? row[i] : -1;
        int32_t doc = -1;
        if (sid >= 0) {
            if (sid < n_sent) doc = s2d[sid];
            else atomicOr(bad, 1);
        }
        bool dup = false;
        for (int j = 0; j < cnt; ++j) dup |= __shfl_sync(0xffffffffu, kept, j) == doc;
        const unsigned peers = __match_any_sync(0xffffffffu, doc);
        const bool ok = doc >= 0 && !dup && (peers & ((1u << lane) - 1)) == 0;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        const int pos = cnt + __popc(m & ((1u << lane) - 1));
        if (ok && pos < k) orow[pos] = doc;
        // lane p takes the doc appended at position p: the (p - cnt)-th surviving lane of this chunk
        const int want = lane - cnt;
        unsigned mm = m;
        for (int s = 0; s < want && mm; ++s) mm &= mm - 1;
        const int src = (want >= 0 && mm) ? __ffs(mm) - 1 : lane;
        const int32_t got = __shfl_sync(0xffffffffu, doc, src);
        if (want >= 0 && want < __popc(m) && lane < k) kept = got;
        cnt = min(k, cnt + __popc(m));
    }
    for (int j = cnt + lane; j < k; j += 32) orow[j] = -1;
}

}  // namespace br

extern "C" int br_dedupe_first_docs(const int64_t* sentence_ids_dev, const int32_t* sentence_to_doc_dev, int64_t n_sentences,
                                    int32_t nq, int32_t n, int32_t k, int64_t* out_docs_dev, void* stream) {
    BR_REQUIRE(sentence_ids_dev && sentence_to_doc_dev && out_docs_dev, BR_ERR_INVALID, "br_dedupe_first_docs: null pointer");
    BR_REQUIRE(nq >= 0 && n >= 0 && k >= 1 && k <= 32, BR_ERR_INVALID, "br_dedupe_first_docs: need nq, n >= 0 and 1 <= k <= 32");
    if (nq == 0) return BR_OK;
    cudaStream_t st = (cudaStream_t)stream;
    br::StreamScratch tmp(st);
    int* d_bad = nullptr;
    BR_TRY(tmp.alloc(&d_bad, 1));
    BR_CUDA(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    br::k_dedupe_first_docs<<<br::blocks_for((int64_t)nq * 32, 128), 128, 0, st>>>(sentence_ids_dev, sentence_to_doc_dev, n_sentences,
                                                                                  nq, n, k, out_docs_dev, d_bad);
    BR_CUDA(cudaGetLastError());
    int bad = 0;
    BR_CUDA(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BR_CUDA(cudaStreamSynchronize(st));
    BR_REQUIRE(!bad, BR_ERR_INVALID, "br_dedupe_first_docs: sentence id outside [0, n_sentences)");
    return BR_OK;
}
