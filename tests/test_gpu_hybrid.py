"""Hybrid retrieval (``document_retrieval_b200.hybrid``): BM25 and dense cosine candidates fused by reciprocal rank
(br_fuse_rrf) or by min-max-normalised exact scores (br_fuse_linear).  Checked bit for bit against a numpy restatement
of both formulas over the GPU's own first-stage lists and components: the BM25 component against ``BM25.exact_scores``,
the cosine component against ``CosineIndex.rerank`` / ``rerank_groups``.  Also the limiting cases, filters and bad
input.  The CPU test at the end checks the numpy restatement against a plain loop."""
import ctypes as C

import numpy as np
import pytest
import torch

from document_retrieval_b200 import synth

gpu = pytest.mark.gpu
BR_ERR_INVALID = -1


# ------------------------------------------------------------------------------------------------ numpy restatement
def first_ranks(lst):
    """{id: 1 + slot of its first occurrence} over the valid ids of one list."""
    r = {}
    for j, x in enumerate(np.asarray(lst).tolist()):
        if x >= 0 and x not in r:
            r[x] = j + 1
    return r


def union_of(b, d):
    u = np.unique(np.r_[np.asarray(b, np.int64), np.asarray(d, np.int64)])
    return u[u >= 0]


def rrf_np(b, d, c=60.0, w_b=1.0, w_d=1.0):
    """-> (union ids ascending, f float64): w_b / (c + r_b) + w_d / (c + r_d), a term omitted when absent."""
    rb, rd = first_ranks(b), first_ranks(d)
    u = union_of(b, d)
    c, w_b, w_d = np.float64(c), np.float64(w_b), np.float64(w_d)
    f = np.empty(u.size, np.float64)
    for i, x in enumerate(u.tolist()):
        if x in rb and x in rd:
            f[i] = w_b / (c + np.float64(rb[x])) + w_d / (c + np.float64(rd[x]))
        elif x in rb:
            f[i] = w_b / (c + np.float64(rb[x]))
        else:
            f[i] = w_d / (c + np.float64(rd[x]))
    return u, f


def linear_np(s_b, s_c, alpha):
    """f = alpha n_b + (1 - alpha) n_c over one union: s_b float64, s_c float32 (NaN: no rows, n_c = 0)."""
    s_b = np.asarray(s_b, np.float64)
    s_c = np.asarray(s_c, np.float32).astype(np.float64)
    has = ~np.isnan(s_c)

    def norm(s, lo, hi):
        return np.zeros_like(s) if hi == lo else (s - lo) / (hi - lo)

    nb = norm(s_b, s_b.min(), s_b.max()) if s_b.size else s_b
    nc = np.zeros_like(s_c)
    if has.any():
        nc[has] = norm(s_c[has], s_c[has].min(), s_c[has].max())
    alpha = np.float64(alpha)
    return alpha * nb + (np.float64(1.0) - alpha) * nc


def top_k(u, f, k):
    """(f desc, id asc), -1 / 0.0 padded to k -> (ids, scores, count)."""
    o = np.lexsort((u, -f))[:k]
    ids = np.full(k, -1, np.int64)
    sc = np.zeros(k, np.float64)
    ids[:o.size], sc[:o.size] = u[o], f[o]
    return ids, sc, o.size


# ------------------------------------------------------------------------------------------------ fixtures
def _setup(seed, n_docs=3000, vocab=1500, nq=24, variant="notebook", dedup=True, d=64, grouped=False):
    """A synth corpus with its BM25 model, a flat or grouped cosine index over the same docs (grouped: 0-4 rows per doc,
    about a fifth of the docs without rows), packed queries (every fifth with an OOV term) and query embeddings."""
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.cosine import CosineIndex
    off, tok = synth.make_corpus(n_docs, vocab, 30, key=(seed,))
    qo, qt, _ = synth.make_queries(off, tok, nq, vocab, key=(seed,), oov_every=5)
    m = BM25.from_token_ids(off, tok, vocab, variant=variant, dedup_query=dedup, device="cuda:0")
    g = torch.Generator().manual_seed(seed)
    if grouped:
        rng = np.random.default_rng(seed)
        sizes = rng.integers(0, 5, n_docs)
        sizes[rng.random(n_docs) < 0.05] = 0
        rg = np.repeat(np.arange(n_docs), sizes)
        ix = CosineIndex(torch.randn(rg.size, d, generator=g), row_group=rg, n_groups=n_docs)
    else:
        ix = CosineIndex(torch.randn(n_docs, d, generator=g))
    qe = torch.randn(nq, d, generator=g).to(torch.bfloat16)
    return m, ix, (qt, qo), qe


def _query(queries, i):
    qt, qo = queries
    return qt[qo[i]:qo[i + 1]].tolist()


def _components(m, ix, queries, qe, unions):
    """Reference components per union: exact BM25 (BM25.exact_scores) and the re-rank cosine (NaN: no rows)."""
    nq = len(unions)
    s_b = [m.exact_scores(_query(queries, i)).cpu().numpy()[u] for i, u in enumerate(unions)]
    W = max(1, max(u.size for u in unions))
    assert W <= 1024
    cand = np.full((nq, W), -1, np.int64)
    for i, u in enumerate(unions):
        cand[i, :u.size] = u
    ids, sims = ix.rerank(qe, cand, W) if ix.row_group is None else ix.rerank_groups(qe, cand, W)
    ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
    s_c = []
    for i, u in enumerate(unions):
        got = dict(zip(ids[i][ids[i] >= 0].tolist(), sims[i][ids[i] >= 0].tolist()))
        s_c.append(np.array([got.get(x, np.nan) for x in u.tolist()], np.float32))
    return s_b, s_c


def _random_lists(rng, nq, nb, nd, n_docs):
    """Query 0: random ids with repeats and -1 slots anywhere; 1: disjoint lists; 2: identical prefixes; 3: partly
    overlapping; 4: both lists empty (all -1); 5: B empty; the rest random."""
    B = rng.integers(-1, n_docs, (nq, nb))
    D = rng.integers(-1, n_docs, (nq, nd))
    B[0, nb // 2:] = B[0, :nb - nb // 2]                               # repeats
    perm = rng.permutation(n_docs)
    B[1], D[1] = perm[:nb], perm[nb:nb + nd]
    w = min(nb, nd)
    B[2, :w] = D[2, :w] = perm[:w]
    B[3], D[3, :nd // 2] = perm[:nb], perm[nb // 2:nb // 2 + nd // 2]
    B[4], D[4] = -1, -1
    B[5] = -1
    return B, D


# ------------------------------------------------------------------------------------------------ 1. RRF bit for bit
@gpu
@pytest.mark.parametrize("nb", [1, 10, 100, 1000])
@pytest.mark.parametrize("nd", [1, 10, 256])
def test_rrf_bit_for_bit(nb, nd):
    from document_retrieval_b200.hybrid import fuse_rrf
    n_docs = 5000
    rng = np.random.default_rng(synth.ROOT_SEED + 13 * nb + nd)
    B, D = _random_lists(rng, 16, nb, nd, n_docs)
    for (c, w_b, w_d) in ((60.0, 1.0, 1.0), (0.0, 2.5, 0.5), (1.5, 0.0, 1.0), (7.0, 1.0, 0.0)):
        for k in (1, 10, min(nb + nd, 1024)):
            ids, sc = fuse_rrf(torch.from_numpy(B), torch.from_numpy(D), n_docs, k, c, (w_b, w_d))
            ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
            for i in range(B.shape[0]):
                ref_ids, ref_sc, cnt = top_k(*rrf_np(B[i], D[i], c, w_b, w_d), k)
                assert np.array_equal(ids[i], ref_ids), (nb, nd, c, k, i)
                assert np.array_equal(sc[i].view(np.int64), ref_sc.view(np.int64)), (nb, nd, c, k, i)
            assert (ids[4] == -1).all() and (sc[4] == 0).all()


@gpu
def test_rrf_ties_break_by_id_and_counts():
    """Disjoint lists with equal weights: rank r in B only ties with rank r in D only; the lower id comes first."""
    from document_retrieval_b200 import _lib
    lib = _lib.load()
    B = torch.tensor([[50, 7, -1, 30, 7]], dtype=torch.int32, device="cuda")
    D = torch.tensor([[3, 60, 20, -1, 99]], dtype=torch.int32, device="cuda")
    ids = torch.empty((1, 12), dtype=torch.int32, device="cuda")
    sc = torch.empty((1, 12), dtype=torch.float64, device="cuda")
    cnt = torch.empty(1, dtype=torch.int32, device="cuda")
    assert lib.br_fuse_rrf(B.data_ptr(), 5, D.data_ptr(), 5, 100, 1, 60.0, 1.0, 1.0, 12, ids.data_ptr(), sc.data_ptr(),
                           cnt.data_ptr(), _lib.stream_ptr(torch.device("cuda"))) == 0
    # ranks: B 50:1 7:2 30:4; D 3:1 60:2 20:3 99:5
    assert ids[0].tolist() == [3, 50, 7, 60, 20, 30, 99] + [-1] * 5
    assert int(cnt[0]) == 7
    assert sc[0, 0] == sc[0, 1] and sc[0, 2] == sc[0, 3]


# ------------------------------------------------------------------------------------------------ 2. linear bit for bit
@gpu
@pytest.mark.parametrize("variant,dedup,grouped", [("notebook", True, False), ("okapi_no_plus1", False, False),
                                                   ("okapi", True, True), ("okapi_no_plus1", True, True),
                                                   ("okapi", False, True)])
def test_linear_bit_for_bit(variant, dedup, grouped):
    """Lists from the GPU's own first stages and random lists (repeats, -1 slots, disjoint / identical / overlapping);
    the components equal exact_scores and the re-rank cosine, the scores the numpy formula over them, the ids the
    lexsort of (-f, id) over the union."""
    from document_retrieval_b200.hybrid import fuse_linear
    m, ix, queries, qe = _setup(31 + 2 * grouped + dedup, variant=variant, dedup=dedup, grouped=grouped)
    nq, n = qe.shape[0], m.corpus_size
    fb, _ = m.retrieve_top_n_batch(queries, 100, positive_only=True)
    fd, _ = ix.topk(qe, 100) if not grouped else ix.topk_groups(qe, 100)
    rng = np.random.default_rng(41)
    rb, rd = _random_lists(rng, nq, 300, 200, n)
    if grouped and variant == "okapi":
        rd[6, :50] = np.flatnonzero(np.bincount(ix.row_group.cpu().numpy(), minlength=n) == 0)[:50]   # docs without rows
    neg = False
    for B, D in ((fb.cpu().numpy(), fd.cpu().numpy()), (rb, rd)):
        unions = [union_of(B[i], D[i]) for i in range(nq)]
        s_b, s_c = _components(m, ix, queries, qe, unions)
        neg |= any((x < 0).any() for x in s_b)
        for alpha in (0.0, 0.3, 0.5, 1.0):
            for k in (1, 10, 500):
                ids, sc, ob, oc = (t.cpu().numpy() for t in fuse_linear(m, ix, queries, qe, B, D, k, alpha))
                for i in range(nq):
                    f = linear_np(s_b[i], s_c[i], alpha)
                    ref_ids, ref_sc, cnt = top_k(unions[i], f, k)
                    assert np.array_equal(ids[i], ref_ids), (alpha, k, i)
                    assert np.array_equal(sc[i].view(np.int64), ref_sc.view(np.int64)), (alpha, k, i)
                    pos = np.searchsorted(unions[i], ids[i, :cnt])
                    assert np.array_equal(ob[i, :cnt].view(np.int64), s_b[i][pos].view(np.int64))
                    np.testing.assert_array_equal(oc[i, :cnt], s_c[i][pos])
                    assert (ob[i, cnt:] == 0).all() and (oc[i, cnt:] == 0).all()
                    if alpha == 1.0:                                    # the order of the exact BM25
                        assert np.array_equal(ids[i, :cnt], top_k(unions[i], s_b[i], k)[0][:cnt])
                    if alpha == 0.0 and not grouped:                   # the order of the re-rank cosine
                        assert np.array_equal(ids[i, :cnt], top_k(unions[i], s_c[i].astype(np.float64), k)[0][:cnt])
    if variant == "okapi_no_plus1":
        assert neg                                                      # negative BM25 scores were covered
    if grouped and variant == "okapi":
        assert np.isnan(s_c[6]).any()                                   # docs without rows were covered


# ------------------------------------------------------------------------------------------------ 3. limiting cases
@gpu
@pytest.mark.parametrize("grouped", [False, True])
def test_limiting_cases(grouped):
    from document_retrieval_b200.hybrid import fuse_rrf, hybrid_search
    m, ix, queries, qe = _setup(57, grouped=grouped)
    n = m.corpus_size
    fb, _, cnt = m.retrieve_top_n_batch(queries, 100, positive_only=True, return_counts=True)
    fd, _ = ix.topk(qe, 50) if not grouped else ix.topk_groups(qe, 50)
    fd = fd.to(torch.int32)
    ids, _ = fuse_rrf(fb, fd, n, 20, weights=(1.0, 0.0))
    for i in range(qe.shape[0]):
        c = min(20, int(cnt[i]))
        assert torch.equal(ids[i, :c], fb[i, :c])                     # BM25 order
    ids, _ = fuse_rrf(fb, fd, n, 50, weights=(0.0, 1.0))
    assert torch.equal(ids, fd)                                       # dense order
    # a query whose terms are all out of vocabulary: an empty BM25 list, a pure dense result
    qt, qo = np.array([m.vocab_size, m.vocab_size + 3], np.int32), np.array([0, 2], np.int32)
    for fusion in ("rrf", "linear"):
        ids, sc = hybrid_search(m, ix, (qt, qo), qe[:1], k=10, n_dense=10, fusion=fusion)
        assert torch.equal(ids[0], fd[0, :10]), fusion


# ------------------------------------------------------------------------------------------------ 4. filters
@gpu
@pytest.mark.parametrize("fusion,grouped", [("rrf", False), ("linear", True), ("linear", False), ("rrf", True)])
def test_filters(fusion, grouped):
    from document_retrieval_b200.hybrid import fuse_linear, fuse_rrf, hybrid_search
    m, ix, queries, qe = _setup(71, grouped=grouped)
    n, nq = m.corpus_size, qe.shape[0]
    rng = np.random.default_rng(72)
    rows = rng.random((3, n)) < np.array([[0.5], [0.05], [0.9]])
    qrow = rng.integers(-1, 3, nq)
    kw = dict(k=20, n_bm25=60, n_dense=40, fusion=fusion, alpha=0.4)
    ids, sc = hybrid_search(m, ix, queries, qe, doc_filter=rows, query_filter=qrow, **kw)
    idn = ids.cpu().numpy()
    for i in range(nq):
        got = idn[i][idn[i] >= 0]
        if qrow[i] >= 0:
            assert rows[qrow[i], got].all(), i
    fb, _ = m.retrieve_top_n_batch(queries, 60, positive_only=True, doc_filter=rows, query_filter=qrow)
    if grouped:
        fd, _ = ix.topk_groups(qe, 40, doc_filter=rows, query_filter=qrow)
    else:
        fd, _ = ix.topk(qe, 40, doc_filter=rows, query_filter=qrow)
    fd = torch.where(fd >= 0, fd, -1)
    if fusion == "rrf":
        ref_ids, ref_sc = fuse_rrf(fb, fd, n, 20)
    else:
        ref_ids, ref_sc = fuse_linear(m, ix, queries, qe, fb, fd, 20, 0.4)[:2]
    assert torch.equal(ids, ref_ids) and torch.equal(sc, ref_sc)
    # an all-ones filter is the unfiltered call, bit for bit
    ids1, sc1 = hybrid_search(m, ix, queries, qe, doc_filter=np.ones(n, bool), **kw)
    ids0, sc0 = hybrid_search(m, ix, queries, qe, **kw)
    assert torch.equal(ids1, ids0) and torch.equal(sc1.view(torch.int64), sc0.view(torch.int64))


# ------------------------------------------------------------------------------------------------ 5. bad input
def _rrf_status(B, D, n_docs, k=10, c=60.0, w=(1.0, 1.0), nq=None):
    from document_retrieval_b200 import _lib
    lib = _lib.load()
    nq = B.shape[0] if nq is None else nq
    ids = torch.empty((max(nq, 1), max(k, 1)), dtype=torch.int32, device="cuda")
    sc = torch.empty((max(nq, 1), max(k, 1)), dtype=torch.float64, device="cuda")
    p = lambda t: None if t is None or t.numel() == 0 else C.c_void_p(t.data_ptr())
    return lib.br_fuse_rrf(p(B), B.shape[1], p(D), D.shape[1], n_docs, nq, c, w[0], w[1], k, p(ids) if nq else None,
                           p(sc) if nq else None, None, _lib.stream_ptr(torch.device("cuda")))


def _linear_status(m, ix, queries, qe, B, D, k=10, alpha=0.5, n_rows=None, nq=None):
    from document_retrieval_b200 import _lib
    lib = _lib.load()
    qt, qo = m._to_device(*m.pack_queries(queries))
    nq = B.shape[0] if nq is None else nq
    ids = torch.empty((max(nq, 1), max(k, 1)), dtype=torch.int32, device="cuda")
    sc = torch.empty((max(nq, 1), max(k, 1)), dtype=torch.float64, device="cuda")
    q = qe.to("cuda").contiguous()
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    return lib.br_fuse_linear(m._h, p(qt), p(qo), nq, qt.numel(), int(m.dedup_query), p(ix.docs), p(ix.inv_norm),
                              ix.n_docs if n_rows is None else n_rows, ix.dim, p(ix.row_group), p(q), p(B), B.shape[1],
                              p(D), D.shape[1], alpha, k, p(ids), p(sc), None, None, None,
                              _lib.stream_ptr(torch.device("cuda")))


@gpu
def test_bad_input():
    from document_retrieval_b200._lib import BRError
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.hybrid import fuse_linear, fuse_rrf, hybrid_search
    m, ix, queries, qe = _setup(91, n_docs=1000, nq=6)
    n = m.corpus_size
    B = torch.randint(-1, n, (6, 20), dtype=torch.int32, device="cuda")
    D = torch.randint(-1, n, (6, 15), dtype=torch.int32, device="cuda")
    assert _rrf_status(B, D, n) == 0
    for v in (-2, n):
        for which in (0, 1):
            bb, dd = B.clone(), D.clone()
            (bb if which == 0 else dd)[3, 4] = v
            assert _rrf_status(bb, dd, n) == BR_ERR_INVALID
            assert _linear_status(m, ix, queries, qe, bb, dd) == BR_ERR_INVALID
            with pytest.raises(BRError):
                fuse_rrf(bb, dd, n)
            with pytest.raises(BRError):
                fuse_linear(m, ix, queries, qe, bb, dd)
    for c, w in ((-1.0, (1.0, 1.0)), (float("nan"), (1.0, 1.0)), (float("inf"), (1.0, 1.0)), (60.0, (0.0, 0.0)),
                 (60.0, (-1.0, 1.0)), (60.0, (1.0, float("inf"))), (60.0, (float("nan"), 1.0))):
        assert _rrf_status(B, D, n, c=c, w=w) == BR_ERR_INVALID, (c, w)
    for k in (0, 1025):
        assert _rrf_status(B, D, n, k=k) == BR_ERR_INVALID
        assert _linear_status(m, ix, queries, qe, B, D, k=k) == BR_ERR_INVALID
    empty = B[:, :0]
    assert _rrf_status(empty, empty, n) == BR_ERR_INVALID                            # nb + nd = 0
    assert _rrf_status(torch.zeros((6, 1025), dtype=torch.int32, device="cuda"), D, n) == BR_ERR_INVALID
    assert _rrf_status(empty, D, n) == 0 and _rrf_status(B, empty, n) == 0
    for a in (-0.1, 1.1, float("nan")):
        assert _linear_status(m, ix, queries, qe, B, D, alpha=a) == BR_ERR_INVALID
        with pytest.raises(BRError):
            fuse_linear(m, ix, queries, qe, B, D, alpha=a)
    assert _linear_status(m, ix, queries, qe, B, D, n_rows=n - 1) == BR_ERR_INVALID   # flat: n_rows != n_docs
    with pytest.raises(ValueError):                                                  # the cosine rows are not the docs
        hybrid_search(m, CosineIndex(torch.randn(n + 1, 64)), queries, qe)
    with pytest.raises(ValueError):
        hybrid_search(m, ix, queries, qe, fusion="sum")
    with pytest.raises(ValueError):
        hybrid_search(m, ix, queries, qe, n_dense=257)
    with pytest.raises(ValueError):
        hybrid_search(m, ix, queries, qe, n_bm25=1025)
    with pytest.raises(ValueError):
        hybrid_search(m, ix, queries, qe[:5])                                        # one embedding per query
    with pytest.raises(ValueError):
        fuse_rrf(B, D[:5], n)
    with pytest.raises(ValueError):
        fuse_rrf(B, D, n, k=0)
    # nq = 0: NULL pointers are fine, and the Python calls return empty tensors
    assert _rrf_status(B[:0], D[:0], n, nq=0) == 0
    for fusion in ("rrf", "linear"):
        ids, sc = hybrid_search(m, ix, [], qe[:0], k=7, fusion=fusion)
        assert ids.shape == (0, 7) and sc.shape == (0, 7)
    ids, sc = fuse_rrf(B, D, n)                                                      # still answers correctly
    ref = [top_k(*rrf_np(B[i].cpu().numpy(), D[i].cpu().numpy()), 10)[0] for i in range(6)]
    assert np.array_equal(ids.cpu().numpy(), np.stack(ref))


# ------------------------------------------------------------------------------------------------ CPU
def test_restatement_matches_a_plain_loop():
    rng = np.random.default_rng(5)
    for _ in range(50):
        nb, nd = int(rng.integers(0, 30)), int(rng.integers(0, 30))
        b, d = rng.integers(-1, 25, nb), rng.integers(-1, 25, nd)
        c, w_b, w_d = float(rng.choice([0.0, 1.0, 60.0])), float(rng.choice([0.0, 1.0, 2.0])), 1.0
        u, f = rrf_np(b, d, c, w_b, w_d)
        want = {}
        for lst, w in ((b, w_b), (d, w_d)):
            seen = set()
            for j, x in enumerate(lst.tolist()):
                if x >= 0 and x not in seen:
                    seen.add(x)
                    want[x] = want.get(x, 0.0) + w / (c + j + 1)
        assert u.tolist() == sorted(want)
        assert f.tolist() == [want[x] for x in u.tolist()]
        ids, sc, cnt = top_k(u, f, 12)
        order = sorted(want, key=lambda x: (-want[x], x))[:12]
        assert ids[:cnt].tolist() == order and (ids[cnt:] == -1).all() and (sc[cnt:] == 0).all()
        # linear: plain loop over the same union
        s_b = rng.standard_normal(u.size) * 3
        s_c = rng.standard_normal(u.size).astype(np.float32)
        s_c[rng.random(u.size) < 0.2] = np.nan
        if u.size > 2:
            s_b[1] = s_b[0]                                               # exact ties
        alpha = float(rng.choice([0.0, 0.25, 1.0]))
        got = linear_np(s_b, s_c, alpha)
        has = [x for x in s_c.tolist() if x == x]
        lo_b, hi_b = (min(s_b), max(s_b)) if u.size else (0, 0)
        lo_c, hi_c = (min(has), max(has)) if has else (0, 0)
        for i in range(u.size):
            nb_ = 0.0 if hi_b == lo_b else (s_b[i] - lo_b) / (hi_b - lo_b)
            x = float(s_c[i])
            nc_ = 0.0 if x != x or hi_c == lo_c else (x - lo_c) / (hi_c - lo_c)
            assert got[i] == alpha * nb_ + (1.0 - alpha) * nc_
