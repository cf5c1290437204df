"""Grouped (document-level) cosine top-k: ``CosineIndex.topk_groups`` ranks groups of embedding rows (a document's
sentences) by their best row's cosine.  Checked against a numpy float32 restatement (normalise, matmul, per-group max,
(score desc, group asc), -1 padding) with the tolerance and near-tie rule of test_gpu_cosine.py, against ``topk`` on
singleton groups, against the reference composition topk(100) + first-seen dedupe (team_run1.py:277-294), and on the
exact fallback, filters, fake shards and bad input.  The two CPU tests at the end check the restatement itself and the
shard split."""
import numpy as np
import pytest
import torch

from document_retrieval_b200 import synth

RTOL, ATOL = 1e-5, 2e-6
gpu = pytest.mark.gpu


def cosine_topk_grouped(docs_f32, q_f32, row_group, n_groups, k, allowed=None):
    """numpy float32 restatement: e/(||e||+1e-10) on both sides, matmul, per-group max over the group's rows, order
    (score desc, group id asc), -1 / 0 padding past the non-empty (allowed) groups.  ``allowed``: bool [Q, G] or None.
    -> (ids int64[Q, k], sims float32[Q, k], group scores float32[Q, G] (-inf: empty or not allowed))"""
    d = np.asarray(docs_f32, np.float32)
    q = np.asarray(q_f32, np.float32)
    d = d / (np.linalg.norm(d, axis=1, keepdims=True) + np.float32(1e-10))
    q = q / (np.linalg.norm(q, axis=1, keepdims=True) + np.float32(1e-10))
    sims = (q @ d.T).astype(np.float32)
    rg = np.asarray(row_group, np.int64)
    gs = np.full((q.shape[0], n_groups), -np.inf, np.float32)
    if rg.size:
        starts = np.flatnonzero(np.r_[True, rg[1:] != rg[:-1]])
        gs[:, rg[starts]] = np.maximum.reduceat(sims, starts, axis=1)
    if allowed is not None:
        gs = np.where(np.asarray(allowed, bool), gs, np.float32(-np.inf))
    ids = np.full((q.shape[0], k), -1, np.int64)
    val = np.zeros((q.shape[0], k), np.float32)
    for i in range(q.shape[0]):
        o = np.lexsort((np.arange(n_groups), -gs[i]))[:k]
        o = o[np.isfinite(gs[i, o])]
        ids[i, :o.size], val[i, :o.size] = o, gs[i, o]
    return ids, val, gs


def _check(ids, sims, ref_ids, ref_sims, gs, nonempty):
    ids, sims = np.asarray(ids), np.asarray(sims)
    for i in range(ids.shape[0]):
        c = int((ref_ids[i] >= 0).sum())
        assert (ids[i, c:] == -1).all() and (sims[i, c:] == 0).all(), i
        got = ids[i, :c]
        assert (got >= 0).all() and nonempty[got].all(), i          # no empty group, ever
        np.testing.assert_allclose(sims[i, :c], ref_sims[i, :c], rtol=RTOL, atol=ATOL)
        if not np.array_equal(got, ref_ids[i, :c]):
            # any difference must be a near-tie in the reference
            np.testing.assert_allclose(gs[i, got], ref_sims[i, :c], rtol=RTOL, atol=ATOL)
            assert len(set(got.tolist())) == c


def _grouped(seed, sizes, d, nq, noise=0.3, qnoise=0.3, n_random_q=0):
    """Rows correlated within a group (group centre + noise), queries = noisy copies of random non-empty group centres
    (+ ``n_random_q`` random queries).  -> (docs bf16, queries bf16, row_group int64, nonempty bool[G])"""
    g = torch.Generator().manual_seed(seed)
    sizes = np.asarray(sizes, np.int64)
    rg = np.repeat(np.arange(sizes.size), sizes)
    centres = torch.randn(sizes.size, d, generator=g)
    docs = (centres[torch.from_numpy(rg)] + noise * torch.randn(rg.size, d, generator=g)).to(torch.bfloat16)
    ne = np.flatnonzero(sizes > 0)
    pick = torch.from_numpy(ne[torch.randint(0, ne.size, (nq,), generator=g).numpy()])
    qs = centres[pick] + qnoise * torch.randn(nq, d, generator=g)
    if n_random_q:
        qs = torch.cat([qs, torch.randn(n_random_q, d, generator=g)])
    return docs, qs.to(torch.bfloat16), rg, sizes > 0


def _ref(docs, qs, rg, n_groups, k, allowed=None):
    return cosine_topk_grouped(docs.float().numpy(), qs.float().numpy(), rg, n_groups, k, allowed)


# ------------------------------------------------------------------------------------------------ 1. singleton groups
@gpu
@pytest.mark.parametrize("n,d,nq,k,kernel", [(20000, 384, 300, 10, 0), (9000, 384, 100, 256, 0), (5000, 1024, 200, 32, 1),
                                             (3000, 1024, 257, 10, 1)])
def test_singleton_groups_equal_topk(n, d, nq, k, kernel):
    """Every row its own group: the same launches, lists and output as topk, bit for bit."""
    from document_retrieval_b200.cosine import CosineIndex, set_cosine_option
    g = torch.Generator().manual_seed(synth.ROOT_SEED + n + k)
    docs = torch.randn(n, d, generator=g).to(torch.bfloat16)
    qs = torch.randn(nq, d, generator=g).to(torch.bfloat16)
    docs[3] = 0
    ix = CosineIndex(docs, doc_base=1000, row_group=torch.arange(n))
    set_cosine_option("kernel", kernel)
    try:
        ids, sims = ix.topk(qs, k)
        gi, gsims = ix.topk_groups(qs, k)
    finally:
        set_cosine_option("kernel", 0)
    assert torch.equal(gi, ids) and torch.equal(gsims, sims)


# ------------------------------------------------------------------------------------------------ 2. random layouts
@gpu
@pytest.mark.parametrize("k", [1, 10, 100, 256])
@pytest.mark.parametrize("d", [64, 200, 768, 1024])
def test_random_layouts_against_reference(d, k):
    """Group sizes 1-40, empty groups in the middle and at the end, one group of 3,000 rows."""
    from document_retrieval_b200.cosine import CosineIndex
    rng = np.random.default_rng(synth.ROOT_SEED + d + k)
    sizes = rng.integers(1, 41, 320)
    sizes[rng.random(320) < 0.1] = 0                                 # empty groups in the middle
    sizes[150] = 3000                                                # one large group
    sizes = np.r_[sizes, np.zeros(7, np.int64)]                     # trailing empty groups
    docs, qs, rg, nonempty = _grouped(d * 1000 + k, sizes, d, 120, n_random_q=40)
    ix = CosineIndex(docs, doc_base=0, row_group=rg, n_groups=sizes.size)
    ids, sims = ix.topk_groups(qs, k)
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, sizes.size, k)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, nonempty)


@gpu
def test_fewer_nonempty_groups_than_k_pad():
    from document_retrieval_b200.cosine import CosineIndex
    sizes = np.array([0, 5, 0, 0, 300, 1, 0, 40, 0])
    docs, qs, rg, nonempty = _grouped(11, sizes, 128, 70)
    ids, sims = CosineIndex(docs, row_group=rg, n_groups=sizes.size, doc_base=5).topk_groups(qs, 10)
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, sizes.size, 10)
    ids = ids.cpu().numpy()
    assert (ids[:, 4:] == -1).all() and (np.sort(ids[:, :4], axis=1) == [6, 9, 10, 12]).all()
    _check(ids - np.where(ids >= 0, 5, 0), sims.cpu().numpy(), ref_ids, ref_sims, gs, nonempty)


# ------------------------------------------------------------------------------------------------ 3. reference composition
@gpu
def test_reference_composition():
    """team_run1.py:277-294: cosine top-100 sentences, then the first 10 distinct parent documents.  Where that yields 10
    documents the grouped top-10 is the same (up to near-ties); where one document's alike sentences fill the 100 rows
    it yields fewer, and the grouped call still returns 10 documents."""
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.sentences import dedupe_sentences_to_docs
    rng = np.random.default_rng(4)
    sizes = rng.integers(1, 30, 900)
    long_docs = [100, 400, 700]
    sizes[long_docs] = 160                                           # long documents of alike sentences
    docs, qs, rg, nonempty = _grouped(12, sizes, 384, 150, noise=0.15, qnoise=0.2, n_random_q=20)
    first_rows = np.cumsum(np.r_[0, sizes])[long_docs]
    qs = torch.cat([qs, docs[first_rows], docs[first_rows + 7]])   # queries that are sentences of the long documents
    ix = CosineIndex(docs, row_group=rg)
    rows, _ = ix.topk(qs, 100)
    comp = dedupe_sentences_to_docs(rows, torch.from_numpy(rg).to(torch.int32).cuda(), 10).cpu().numpy()
    ids, sims = ix.topk_groups(qs, 10)
    ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, sizes.size, 10)
    _check(ids, sims, ref_ids, ref_sims, gs, nonempty)
    short = (comp < 0).any(axis=1)
    assert short.sum() >= 6, "the data must hold queries whose top-100 rows name fewer than 10 documents"
    assert (ids[short] >= 0).all()
    for i in np.flatnonzero(~short):
        if not np.array_equal(ids[i], comp[i]):
            # the composition's documents differ only where reference group scores are near-tied
            np.testing.assert_allclose(gs[i, comp[i]], ref_sims[i], rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------ 4. warm-up bound
@gpu
def test_warmup_never_overflows_at_k256():
    """k = 256 over documents of 20 near-duplicate sentences at d = 1032: the exact gather pass supports d <= 1024 only,
    so the call fails with BR_ERR_UNSUPPORTED if any query overflowed its candidate list.  It must not."""
    from document_retrieval_b200.cosine import CosineIndex
    sizes = np.full(600, 20)
    docs, qs, rg, nonempty = _grouped(13, sizes, 1032, 80, noise=0.02, qnoise=0.3, n_random_q=20)
    ids, sims = CosineIndex(docs, row_group=rg).topk_groups(qs, 256)
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, sizes.size, 256)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, nonempty)


# ------------------------------------------------------------------------------------------------ 5. exact fallback
@gpu
def test_overflow_fallback_is_exact():
    """2,000 identical rows in 2,000 groups and one group of 1,500 copies of another row: queries equal to them overflow
    the candidate lists (more than 64 of them: several sub-batches of the exact pass) and are answered exactly, ties by
    group id."""
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(14)
    d = 128
    a = torch.randn(1000, d, generator=g)
    x, y = torch.randn(1, d, generator=g), torch.randn(1, d, generator=g)
    b = torch.randn(1000, d, generator=g)
    docs = torch.cat([a, x.repeat(2000, 1), y.repeat(1500, 1), b]).to(torch.bfloat16)
    rg = np.r_[np.arange(1000), 1000 + np.arange(2000), np.full(1500, 3000), 3001 + np.arange(1000)]
    qs = torch.cat([x.repeat(70, 1), y.repeat(70, 1), torch.randn(30, d, generator=g)]).to(torch.bfloat16)
    ids, sims = CosineIndex(docs, row_group=rg, doc_base=7).topk_groups(qs, 10)
    ids, sims = ids.cpu().numpy() - 7, sims.cpu().numpy()
    assert (ids[:70] == np.arange(1000, 1010)).all()                # exact ties by group id
    assert (ids[70:140, 0] == 3000).all()
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, 4001, 10)
    _check(ids, sims, ref_ids, ref_sims, gs, np.ones(4001, bool))


# ------------------------------------------------------------------------------------------------ 6. filters
@gpu
@pytest.mark.parametrize("kernel", [0, 1])
def test_filters_over_groups(kernel):
    from document_retrieval_b200.cosine import CosineIndex, set_cosine_option
    rng = np.random.default_rng(15)
    sizes = rng.integers(0, 25, 1500)
    G = sizes.size
    docs, qs, rg, nonempty = _grouped(15, sizes, 256, 200, n_random_q=30)
    nq = qs.shape[0]
    lang = rng.integers(0, 7, G)
    rows = np.stack([rng.random(G) < 0.5, rng.random(G) < 0.01] + [lang == i for i in range(7)]
                    + [np.zeros(G, bool)])
    rows[-1, [3, 700, G - 1]] = True                                  # 3 allowed groups, fewer than k: -1 padding
    qrow = (rng.integers(-1, rows.shape[0], nq)).astype(np.int32)
    qrow[:5] = rows.shape[0] - 1
    ix = CosineIndex(docs, row_group=rg, n_groups=G)
    set_cosine_option("kernel", kernel)
    try:
        ids, sims = ix.topk_groups(qs, 10, doc_filter=rows, query_filter=qrow)
        ids_u, sims_u = ix.topk_groups(qs, 10)
        ids_1, sims_1 = ix.topk_groups(qs, 10, doc_filter=np.ones(G, bool))
    finally:
        set_cosine_option("kernel", 0)
    allowed = np.where((qrow >= 0)[:, None], rows[np.maximum(qrow, 0)], True)
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, G, 10, allowed)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, nonempty)
    assert torch.equal(ids_1, ids_u) and torch.equal(sims_1, sims_u)
    unf = torch.from_numpy(qrow < 0).cuda()
    assert torch.equal(ids[unf], ids_u[unf]) and torch.equal(sims[unf], sims_u[unf])
    assert (ids[:5, 3:] == -1).all()


# ------------------------------------------------------------------------------------------------ 7. fake shards
@gpu
@pytest.mark.parametrize("world", [2, 5])
def test_fake_shards_equal_single_index(world):
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.sharded import ShardedCosineIndex, group_shard_bounds, local_filter_slice, merge_topk_cuda
    rng = np.random.default_rng(16)
    sizes = rng.integers(0, 40, 600)
    G = sizes.size
    docs, qs, rg, nonempty = _grouped(16, sizes, 192, 150, noise=0.6, n_random_q=30)
    filt = np.stack([rng.random(G) < 0.3, np.ones(G, bool)])
    qrow = (np.arange(qs.shape[0]) % 3 - 1).astype(np.int32)
    ix = CosineIndex(docs, row_group=rg, n_groups=G)
    for kw in ({}, dict(doc_filter=filt, query_filter=qrow)):
        ids1, s1 = ix.topk_groups(qs, 10, **kw)
        parts = []
        for lo, hi in group_shard_bounds(rg, world):
            assert hi > lo and (lo == 0 or rg[lo] != rg[lo - 1])
            g_lo, g_hi = int(rg[lo]), int(rg[hi - 1]) + 1
            pkw = {} if not kw else dict(doc_filter=local_filter_slice(filt, g_lo, g_hi - g_lo), query_filter=qrow)
            parts.append(CosineIndex(docs[lo:hi], row_group=rg[lo:hi] - g_lo, doc_base=g_lo).topk_groups(qs, 10, **pkw))
        ids_m, sc_m = merge_topk_cuda(torch.stack([p[0] for p in parts]), torch.stack([p[1].double() for p in parts]), 10)
        assert torch.equal(ids_m, ids1) and torch.equal(sc_m, s1.double())
        one = ShardedCosineIndex(docs, 0, row_group=rg, n_groups=G)   # one rank: the global ids are its own
        i2, s2 = one.topk_groups(qs, 10, **kw)
        assert torch.equal(i2, ids1) and torch.equal(s2, s1.double())
    ids, sims = ix.topk_groups(qs, 10)
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, G, 10)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, nonempty)


# ------------------------------------------------------------------------------------------------ 8. bad input
@gpu
def test_bad_input():
    from document_retrieval_b200._lib import BRError
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(17)
    docs = torch.randn(3000, 64, generator=g).to(torch.bfloat16)
    qs = torch.randn(9, 64, generator=g).to(torch.bfloat16)
    rg = np.repeat(np.arange(300), 10)
    dec = rg.copy()
    dec[1500], dec[1501] = dec[1501], dec[1500] - 1                   # decreasing at 1501
    with pytest.raises(BRError):
        CosineIndex(docs, row_group=dec).topk_groups(qs, 10)
    with pytest.raises(BRError):                                     # a value >= n_groups
        CosineIndex(docs, row_group=rg, n_groups=299).topk_groups(qs, 10)
    neg = rg.copy()
    neg[:10] = -1
    with pytest.raises(BRError):
        CosineIndex(docs, row_group=neg).topk_groups(qs, 10)
    with pytest.raises(ValueError):                                  # length does not match the rows
        CosineIndex(docs, row_group=rg[:-1])
    ix = CosineIndex(docs, row_group=rg, n_groups=310)
    with pytest.raises(ValueError):                                  # filter over rows, not groups
        ix.topk_groups(qs, 10, doc_filter=np.ones(3000, bool))
    with pytest.raises(BRError):                                     # query_filter row out of range
        ix.topk_groups(qs, 10, doc_filter=np.ones((2, 310), bool), query_filter=np.array([0, 1, 2, 0, 0, 0, 0, 0, 0]))
    for k in (0, 257):
        with pytest.raises(BRError):
            ix.topk_groups(qs, k)
    with pytest.raises(ValueError):
        CosineIndex(docs).topk_groups(qs, 10)
    ids, sims = ix.topk_groups(qs, 10)                               # the index still answers correctly
    ref_ids, ref_sims, gs = _ref(docs, qs, rg, 310, 10)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, np.arange(310) < 300)


# ------------------------------------------------------------------------------------------------ CPU
def test_reference_restatement_matches_a_plain_loop():
    rng = np.random.default_rng(18)
    sizes = np.r_[0, rng.integers(0, 6, 40), 0, 0]
    rg = np.repeat(np.arange(sizes.size), sizes)
    docs = rng.standard_normal((rg.size, 16)).astype(np.float32)
    docs[5:9] = docs[4]                                               # exact ties across rows
    qs = np.r_[docs[4:5], rng.standard_normal((6, 16)).astype(np.float32)]
    allowed = rng.random((qs.shape[0], sizes.size)) < 0.7
    for alw in (None, allowed):
        ids, val, gs = cosine_topk_grouped(docs, qs, rg, sizes.size, 12, alw)
        dn = docs / (np.linalg.norm(docs, axis=1, keepdims=True) + np.float32(1e-10))
        qn = qs / (np.linalg.norm(qs, axis=1, keepdims=True) + np.float32(1e-10))
        s = qn @ dn.T
        for i in range(qs.shape[0]):
            best = {}
            for r, gid in enumerate(rg):
                if alw is None or alw[i, gid]:
                    best[gid] = max(best.get(gid, -np.inf), s[i, r])
            want = sorted(best, key=lambda x: (-best[x], x))[:12]
            assert ids[i, :len(want)].tolist() == want and (ids[i, len(want):] == -1).all()
            np.testing.assert_allclose(val[i, :len(want)], [best[x] for x in want], rtol=1e-6)


def test_group_shard_bounds_keep_groups_whole():
    from document_retrieval_b200.sharded import group_shard_bounds, shard_bounds
    rng = np.random.default_rng(19)
    rg = np.repeat(np.arange(500), rng.integers(0, 30, 500))
    for world in (1, 2, 3, 5, 8):
        b = group_shard_bounds(rg, world)
        assert len(b) == world and b[0][0] == 0 and b[-1][1] == rg.size
        assert all(b[r][1] == b[r + 1][0] for r in range(world - 1))
        for lo, hi in b:
            assert lo == 0 or lo == rg.size or rg[lo] != rg[lo - 1]
        assert all(b[r][0] >= shard_bounds(rg.size, world)[r][0] for r in range(world))
    big = np.r_[np.zeros(90, np.int64), np.arange(1, 11)]            # one group of 90 rows in 100
    assert group_shard_bounds(big, 4) == [(0, 90), (90, 90), (90, 90), (90, 100)]
