"""GPU: dense cosine top-k (tcgen05 GEMM, fused norm + top-k) and candidate re-rank against the
oracle restatement of team_run1.py:270-282 and its golden fixture.  Tolerance (north_star): cosine
scores within 1e-5 relative in fp32 (plus 2e-6 absolute for values near zero); ids identical except
where two reference scores are closer than that tolerance."""
import numpy as np
import pytest
import torch

from oracle import bm25_oracle as orc
from document_retrieval_b200 import synth

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-5, 2e-6


def _check(ids, sims, docs_f32, q_f32, k):
    ref_ids, ref_sims = orc.cosine_topk(docs_f32, q_f32, k)
    d = torch.as_tensor(docs_f32)
    dn = d / (d.norm(dim=1, keepdim=True) + 1e-10)
    qn = torch.as_tensor(q_f32)
    qn = qn / (qn.norm(dim=1, keepdim=True) + 1e-10)
    full = (qn @ dn.T).numpy()
    np.testing.assert_allclose(sims, ref_sims, rtol=RTOL, atol=ATOL)
    for i in range(ids.shape[0]):
        if not np.array_equal(ids[i], ref_ids[i]):
            # any difference must be a near-tie in the reference
            np.testing.assert_allclose(full[i, ids[i]], ref_sims[i], rtol=RTOL, atol=ATOL)
            assert len(set(ids[i].tolist())) == k


def test_cosine_topk_golden(golden):
    from document_retrieval_b200.cosine import CosineIndex
    g = golden("cosine_small")
    docs = torch.from_numpy(g["docs_bf16"]).view(torch.bfloat16)
    qs = torch.from_numpy(g["queries_bf16"]).view(torch.bfloat16)
    ix = CosineIndex(docs)
    ids, sims = ix.topk(qs, 10)
    ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
    np.testing.assert_allclose(sims, g["top_sims"], rtol=RTOL, atol=ATOL)
    assert np.array_equal(ids, g["top_ids"])


@pytest.mark.parametrize("n,d,nq,k", [(5000, 768, 300, 10), (777, 128, 5, 3), (130, 64, 257, 10), (20000, 384, 64, 32),
                                      (3000, 200, 500, 10),      # d not a multiple of the 64-wide k-block (TMA zero fill)
                                      (2000, 1024, 300, 10),     # d > 768: the query block does not fit -> multicast kernel
                                      (40000, 96, 1000, 5),      # several query blocks
                                      (58000, 96, 1000, 5)])     # a launch across two L2 windows x several query blocks
def test_cosine_topk_random(n, d, nq, k):
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(synth.ROOT_SEED + n)
    docs = torch.randn(n, d, generator=g).to(torch.bfloat16)
    qs = torch.randn(nq, d, generator=g).to(torch.bfloat16)
    docs[3] = 0                                              # zero-norm doc: e/(0+1e-10) = 0
    ix = CosineIndex(docs, doc_base=1000)
    ids, sims = ix.topk(qs, k)
    _check(ids.cpu().numpy() - 1000, sims.cpu().numpy(), docs.float().numpy(), qs.float().numpy(), k)


@pytest.mark.parametrize("n,d,nq,k", [(9000, 320, 700, 10), (5000, 768, 300, 10), (777, 128, 5, 3), (130, 64, 257, 10),
                                      (20000, 384, 64, 32),
                                      (3000, 200, 500, 10),      # d not a multiple of the 64-wide k-block (TMA zero fill)
                                      (40000, 96, 1000, 5),
                                      (58000, 96, 1000, 5)])     # a launch across two L2 windows x several query blocks
def test_cosine_kernel_variants_agree(n, d, nq, k):
    """The two production GEMM kernels, query-stationary CTA pairs (the default at d <= 768) and 2-CTA multicast (the
    kernel for d > 768, forced here), return the same ids and bit-identical similarities: same K order of accumulation
    per element."""
    from document_retrieval_b200.cosine import CosineIndex, set_cosine_option
    g = torch.Generator().manual_seed(99 + n)
    docs = torch.randn(n, d, generator=g).to(torch.bfloat16)
    qs = torch.randn(nq, d, generator=g).to(torch.bfloat16)
    ix = CosineIndex(docs)
    ids0, s0 = ix.topk(qs, k)
    try:
        set_cosine_option("kernel", 1)
        ids1, s1 = ix.topk(qs, k)
    finally:
        set_cosine_option("kernel", 0)
    assert torch.equal(ids0, ids1) and torch.equal(s0, s1)


def test_cosine_rerank_of_bm25_candidates():
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.cosine import CosineIndex, rerank_bm25_with_cosine
    c = synth.make_config("C1", scale=0.3)
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    g = torch.Generator().manual_seed(7)
    emb = torch.randn(c["n_docs"], 768, generator=g).to(torch.bfloat16)
    qe = torch.randn(c["q_offsets"].size - 1, 768, generator=g).to(torch.bfloat16)
    ix = CosineIndex(emb)
    ids, sims = rerank_bm25_with_cosine(m, ix, (c["q_terms"], c["q_offsets"]), qe, n_candidates=200, k=10)
    ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
    cand, _ = m.retrieve_top_n_batch((c["q_terms"], c["q_offsets"]), 200)
    cand = cand.cpu().numpy()
    e32, q32 = emb.float().numpy(), qe.float().numpy()
    for i in range(0, ids.shape[0], 17):
        cc = cand[i][cand[i] >= 0]
        ri, rs = orc.cosine_topk(e32[cc], q32[i:i + 1], 10)
        np.testing.assert_allclose(sims[i], rs[0], rtol=RTOL, atol=ATOL)
        assert set(ids[i].tolist()) <= set(cc.tolist())
        if not np.array_equal(ids[i], cc[ri[0]]):
            assert np.allclose(np.sort(sims[i]), np.sort(rs[0]), rtol=RTOL, atol=ATOL)


def test_cosine_massive_ties_are_answered_exactly():
    """2,000 identical embedding rows: a query equal to them has 2,000 candidates tied at the top - more than the filter's
    1,024-slot lists hold - and must still get the exact answer (lowest row ids first), like every other query."""
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(5)
    docs = torch.randn(6000, 128, generator=g).to(torch.bfloat16)
    dup = torch.arange(1000, 6000, 2)[:2000]
    docs[dup] = docs[999].clone()
    qs = torch.cat([docs[999:1000], torch.randn(40, 128, generator=g).to(torch.bfloat16)])
    ids, sims = CosineIndex(docs).topk(qs, 10)
    ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
    want = np.sort(np.concatenate([[999], dup.numpy()]))[:10]
    assert np.array_equal(ids[0], want)
    np.testing.assert_allclose(sims[0], 1.0, rtol=1e-5)
    _check(ids[1:], sims[1:], docs.float().numpy(), qs[1:].float().numpy(), 10)


def test_cosine_topk_overflow_fallback_for_many_queries():
    """ADVICE r1: more than 64 queries whose candidates overflow the filter lists in one launch.  (a) 100 queries equal to a
    row that is duplicated 2,000 times; (b) a corpus SORTED by similarity to the query direction, so that every launch sees
    only rows better than everything before it.  Both must be answered exactly (gather-pass fallback in sub-batches)."""
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(synth.ROOT_SEED + 77)
    n, d, k = 30000, 64, 10
    docs = torch.randn(n, d, generator=g).to(torch.bfloat16)
    docs[5000:7000] = docs[123]                                   # 2,001 identical rows
    qs = docs[123:124].repeat(100, 1).clone()
    qs[50:] += (0.01 * torch.randn(50, d, generator=g)).to(torch.bfloat16)
    ix = CosineIndex(docs)
    ids, sims = ix.topk(qs, k)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), docs.float().numpy(), qs.float().numpy(), k)
    assert ids[0].cpu().tolist() == [123] + list(range(5000, 5009))          # exact ties by row id
    # (b) rows sorted by ascending cosine to a direction; 80 queries close to that direction
    v = torch.randn(d, generator=g)
    base = torch.randn(n, d, generator=g)
    order = torch.argsort((base / base.norm(dim=1, keepdim=True)) @ (v / v.norm()))
    docs2 = base[order].to(torch.bfloat16)
    qs2 = (v[None, :] + 0.05 * torch.randn(80, d, generator=g)).to(torch.bfloat16)
    ix2 = CosineIndex(docs2)
    ids2, sims2 = ix2.topk(qs2, k)
    _check(ids2.cpu().numpy(), sims2.cpu().numpy(), docs2.float().numpy(), qs2.float().numpy(), k)
