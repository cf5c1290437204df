"""Grouped cosine re-rank: ``CosineIndex.rerank_groups`` scores each query's candidate groups (a BM25 document's
sentences) by their best row's cosine.  Checked bit for bit against ``rerank`` over the expanded rows followed by a
per-group max, against ``rerank`` on singleton groups, against ``topk_groups`` when every group is a candidate, on
padding, on the BM25 -> sentence pipeline against a numpy float32 restatement, on fake shards and on bad input.  The CPU
test at the end checks the file's numpy restatement against a plain loop."""
import ctypes as C

import numpy as np
import pytest
import torch

from document_retrieval_b200 import synth

RTOL, ATOL = 1e-5, 2e-6
gpu = pytest.mark.gpu
BR_ERR_INVALID, BR_ERR_UNSUPPORTED = -1, -4


def rerank_grouped_np(docs_f32, q_f32, row_group, n_groups, cand, k):
    """numpy float32 restatement: e/(||e||+1e-10) on both sides, matmul, per-group max over the group's rows, restricted
    to each query's distinct candidates (-1 skipped), order (score desc, group id asc), -1 / 0 padding past the
    non-empty candidates.  -> (ids int64[Q, k], sims float32[Q, k], group scores float32[Q, G] (-inf: empty))"""
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
    ids = np.full((q.shape[0], k), -1, np.int64)
    val = np.zeros((q.shape[0], k), np.float32)
    for i in range(q.shape[0]):
        c = np.unique(np.asarray(cand[i], np.int64))
        c = c[c >= 0]
        c = c[np.isfinite(gs[i, c])]
        o = c[np.lexsort((c, -gs[i, c]))][:k]
        ids[i, :o.size], val[i, :o.size] = o, gs[i, o]
    return ids, val, gs


def _check(ids, sims, ref_ids, ref_sims, gs, nonempty):
    """The tolerance and near-tie rule of the grouped top-k tests."""
    ids, sims = np.asarray(ids), np.asarray(sims)
    for i in range(ids.shape[0]):
        c = int((ref_ids[i] >= 0).sum())
        assert (ids[i, c:] == -1).all() and (sims[i, c:] == 0).all(), i
        got = ids[i, :c]
        assert (got >= 0).all() and nonempty[got].all(), i
        np.testing.assert_allclose(sims[i, :c], ref_sims[i, :c], rtol=RTOL, atol=ATOL)
        if not np.array_equal(got, ref_ids[i, :c]):
            np.testing.assert_allclose(gs[i, got], ref_sims[i, :c], rtol=RTOL, atol=ATOL)
            assert len(set(got.tolist())) == c


def _grouped(seed, sizes, d, nq, noise=0.3, qnoise=0.3):
    """Rows = group centre + noise; queries = noisy copies of random non-empty group centres.
    -> (docs bf16, queries bf16, row_group int64, nonempty bool[G])"""
    g = torch.Generator().manual_seed(seed)
    sizes = np.asarray(sizes, np.int64)
    rg = np.repeat(np.arange(sizes.size), sizes)
    centres = torch.randn(sizes.size, d, generator=g)
    docs = (centres[torch.from_numpy(rg)] + noise * torch.randn(rg.size, d, generator=g)).to(torch.bfloat16)
    ne = np.flatnonzero(sizes > 0)
    pick = torch.from_numpy(ne[torch.randint(0, ne.size, (nq,), generator=g).numpy()])
    qs = centres[pick] + qnoise * torch.randn(nq, d, generator=g)
    return docs, qs.to(torch.bfloat16), rg, sizes > 0


def _layout(rng, n_groups, big=3000):
    """Group sizes 1-40, about 10 % empty, several 1-row groups, one group of ``big`` rows; group 0 has rows."""
    sizes = rng.integers(1, 41, n_groups)
    sizes[rng.random(n_groups) < 0.1] = 0
    sizes[rng.random(n_groups) < 0.1] = 1
    sizes[0] = 3
    sizes[n_groups // 3] = big
    return np.r_[sizes, 0, 0]                                        # trailing empty groups


def _via_rows(ix, qs, cand, k):
    """The per-row composition: every expanded row's cosine from ``rerank`` (chunks of <= 1024 rows with k = the chunk
    width, so every row comes back), the max per group, order (score desc, group asc), -1 / 0 padding."""
    dev = ix.device
    rg = ix.row_group.to(torch.int64)
    G, n = ix.n_groups, ix.n_docs
    cand = torch.as_tensor(cand).to(dev, torch.int64)
    Q = cand.shape[0]
    member = torch.zeros((Q, G + 1), dtype=torch.bool, device=dev)     # distinct candidates per query (column G: -1)
    member.scatter_(1, torch.where(cand >= 0, cand, G), True)
    member = member[:, :G]
    row_on = member[:, rg]                                             # [Q, n] rows of the query's candidates
    cnt = row_on.sum(1)
    width = max(1, int(cnt.max()))
    rows = torch.full((Q, width), -1, dtype=torch.int32, device=dev)
    pos = torch.cumsum(row_on.to(torch.int64), 1) - 1
    qi, ri = torch.nonzero(row_on, as_tuple=True)
    rows[qi, pos[qi, ri]] = ri.to(torch.int32)
    row_sim = torch.full((Q, n), -float("inf"), dtype=torch.float32, device=dev)
    for j in range(0, width, 1024):
        part = rows[:, j:j + 1024].contiguous()
        ids, sims = ix.rerank(qs, part, part.shape[1])
        ok = ids >= 0
        qq = torch.arange(Q, device=dev)[:, None].expand_as(ids)
        row_sim[qq[ok], ids[ok].to(torch.int64)] = sims[ok]
    gmax = torch.full((Q, G), -float("inf"), dtype=torch.float32, device=dev)
    gmax.scatter_reduce_(1, rg[None].expand(Q, n), row_sim, "amax")
    score, order = torch.sort(gmax, dim=1, descending=True, stable=True)   # ties: lower group first
    score, order = score[:, :k], order[:, :k]
    if score.shape[1] < k:
        score = torch.cat([score, torch.full((Q, k - score.shape[1]), -float("inf"), device=dev)], 1)
        order = torch.cat([order, torch.zeros((Q, k - order.shape[1]), dtype=order.dtype, device=dev)], 1)
    valid = score > -float("inf")
    return (torch.where(valid, order, -1).to(torch.int32),
            torch.where(valid, score, torch.zeros_like(score)))


def _bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _candidates(rng, Q, c, G, sizes):
    """Random ids in [-1, G) with repeats; query 0 lists only empty groups and -1; query 1 repeats the large group."""
    cand = rng.integers(-1, G, (Q, c))
    empty = np.flatnonzero(sizes == 0)
    cand[0] = np.where(rng.random(c) < 0.5, -1, empty[rng.integers(0, empty.size, c)])
    cand[1, ::2] = int(np.argmax(sizes))
    return cand


# ------------------------------------------------------------------------------------------------ 1. bit identity
@gpu
@pytest.mark.parametrize("d", [8, 256, 264, 512, 520, 768, 1024])
def test_bit_identical_to_row_rerank_and_group_max(d):
    """Random layouts with empty, 1-row and 3,000-row groups; c = 1 / 7 / 1000 / 5000 (duplicates, -1 slots, lists of
    only empty groups); k = 1 / 10 / 100 / 1024: ids and the sims' bits equal the per-row composition."""
    from document_retrieval_b200.cosine import CosineIndex
    rng = np.random.default_rng(synth.ROOT_SEED + d)
    sizes = _layout(rng, 600)
    G = sizes.size
    docs, qs, rg, _ = _grouped(d, sizes, d, 12)
    docs[5] = 0                                                      # a zero row
    ix = CosineIndex(docs, row_group=rg, n_groups=G)
    for c, k in ((1, 1), (1, 10), (7, 1), (7, 10), (1000, 10), (1000, 100), (1000, 1024), (5000, 10), (5000, 1024)):
        cand = _candidates(rng, qs.shape[0], c, G, sizes)
        ids, sims = ix.rerank_groups(qs, cand, k)
        ref_ids, ref_sims = _via_rows(ix, qs, cand, k)
        assert torch.equal(ids, ref_ids), (d, c, k)
        assert _bits_equal(sims, ref_sims), (d, c, k)
        assert (ids[0] == -1).all() and (sims[0] == 0).all()           # only empty groups: all padding


# ------------------------------------------------------------------------------------------------ 2. singleton groups
@gpu
@pytest.mark.parametrize("d,k", [(256, 10), (768, 1024), (1024, 100)])
def test_singleton_groups_equal_rerank(d, k):
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(synth.ROOT_SEED + 7 * d + k)
    n = 20000
    docs = torch.randn(n, d, generator=g).to(torch.bfloat16)
    qs = torch.randn(40, d, generator=g).to(torch.bfloat16)
    docs[3] = 0
    cand = torch.randint(-1, n, (40, 1500), generator=g)
    cand[:, 100:200] = cand[:, :100]                                 # repeats
    ix = CosineIndex(docs, row_group=torch.arange(n))
    ids, sims = ix.rerank(qs, cand, k)
    gi, gs = ix.rerank_groups(qs, cand, k)
    assert torch.equal(gi, ids) and _bits_equal(gs, sims)


# ------------------------------------------------------------------------------------------------ 3. brute-force grouped
@gpu
@pytest.mark.parametrize("k", [1, 10, 100, 256])
def test_all_groups_as_candidates_match_topk_groups(k):
    from document_retrieval_b200.cosine import CosineIndex
    rng = np.random.default_rng(synth.ROOT_SEED + 300 + k)
    sizes = _layout(rng, 400)
    G = sizes.size
    docs, qs, rg, nonempty = _grouped(300 + k, sizes, 384, 60)
    ix = CosineIndex(docs, row_group=rg, n_groups=G)
    ti, ts = ix.topk_groups(qs, k)
    ids, sims = ix.rerank_groups(qs, np.tile(np.arange(G), (qs.shape[0], 1)), k)
    ti, ts = ti.cpu().numpy(), ts.cpu().numpy()
    gs = rerank_grouped_np(docs.float().numpy(), qs.float().numpy(), rg, G, np.tile(np.arange(G), (qs.shape[0], 1)), k)[2]
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ti, ts, gs, nonempty)


# ------------------------------------------------------------------------------------------------ 4. padding
@gpu
def test_fewer_candidates_than_k_pad():
    from document_retrieval_b200.cosine import CosineIndex
    sizes = np.array([4, 0, 5, 0, 0, 300, 1, 0, 40, 0])
    docs, qs, rg, nonempty = _grouped(41, sizes, 128, 20)
    ix = CosineIndex(docs, row_group=rg, n_groups=sizes.size)
    cand = np.tile(np.array([5, 1, 2, -1, 5, 9, 6, 3, 2, 8, -1]), (20, 1))   # 5 distinct non-empty: 2, 5, 6, 8 and dup
    ids, sims = ix.rerank_groups(qs, cand, 10)
    ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
    assert (np.sort(ids[:, :4], axis=1) == [2, 5, 6, 8]).all()
    assert (ids[:, 4:] == -1).all() and (sims[:, 4:] == 0).all()
    ref_ids, ref_sims, gs = rerank_grouped_np(docs.float().numpy(), qs.float().numpy(), rg, sizes.size, cand, 10)
    _check(ids, sims, ref_ids, ref_sims, gs, nonempty)


# ------------------------------------------------------------------------------------------------ 5. pipeline
@gpu
def test_bm25_to_sentences_pipeline():
    """BM25 top-1000 documents, each scored by its best sentence: the numpy restatement over the oracle's BM25 ranking."""
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.cosine import CosineIndex, rerank_bm25_with_sentences
    from oracle import bm25_oracle as orc
    c = synth.make_config("C1", scale=0.25)
    n_docs = len(c["doc_offsets"]) - 1
    assert n_docs > 1000
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], device="cuda:0")
    rng = np.random.default_rng(51)
    sizes = (1 + np.floor(31 * rng.random(n_docs) ** 3)).astype(np.int64)
    nq = 40
    docs, _, rg, nonempty = _grouped(51, sizes, 96, 1)
    qe = torch.randn(nq, 96, generator=torch.Generator().manual_seed(52)).to(torch.bfloat16)
    ix = CosineIndex(docs, row_group=rg, n_groups=n_docs)
    qt, qo = c["q_terms"], c["q_offsets"]
    sub = (qt[:qo[nq]], qo[:nq + 1])
    ids, sims = rerank_bm25_with_sentences(m, ix, sub, qe, n_candidates=1000, k=10)
    oix = orc.build_index(c["doc_offsets"], c["token_ids"], c["vocab"])
    cand = np.stack([orc.topk_canonical(orc.get_scores(oix, qt[qo[i]:qo[i + 1]]), 1000)[0] for i in range(nq)])
    ref_ids, ref_sims, gs = rerank_grouped_np(docs.float().numpy(), qe.float().numpy(), rg, n_docs, cand, 10)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, nonempty)
    with pytest.raises(ValueError):                                  # groups that are not the BM25 documents
        rerank_bm25_with_sentences(m, CosineIndex(docs, row_group=rg, n_groups=n_docs + 1), sub, qe)


# ------------------------------------------------------------------------------------------------ 6. fake shards
@gpu
@pytest.mark.parametrize("world", [2, 5])
def test_fake_shards_equal_single_index(world):
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.sharded import ShardedCosineIndex, group_shard_bounds, local_group_candidates, merge_topk_cuda
    rng = np.random.default_rng(61 + world)
    sizes = _layout(rng, 500, big=400)
    G = sizes.size
    docs, qs, rg, _ = _grouped(61, sizes, 192, 30, noise=0.6)
    bounds = group_shard_bounds(rg, world)
    cuts = [0] + [int(rg[lo]) for lo, _ in bounds[1:]] + [G]          # shard r owns groups [cuts[r], cuts[r + 1])
    cand = rng.integers(-1, G, (qs.shape[0], 700))
    for r in range(1, world):                                        # ids on both sides of every shard edge
        cand[:, r] = cuts[r] - 1
        cand[:, world + r] = cuts[r]
    ix = CosineIndex(docs, row_group=rg, n_groups=G)
    for k in (10, 100):
        ids1, s1 = ix.rerank_groups(qs, cand, k)
        parts, owned = [], 0
        for r, (lo, hi) in enumerate(bounds):
            g_lo, g_hi = cuts[r], cuts[r + 1]
            local, n_own = local_group_candidates(cand, g_lo, g_hi - g_lo)
            owned += n_own
            sh = CosineIndex(docs[lo:hi], row_group=rg[lo:hi] - g_lo, n_groups=g_hi - g_lo, group_base=g_lo)
            i, s = sh.rerank_groups(qs, local, k)
            parts.append((torch.where(i >= 0, i.to(torch.int64) + g_lo, -1), s.double()))
        assert owned == int((cand >= 0).sum())
        ids_m, sc_m = merge_topk_cuda(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]), k)
        assert torch.equal(ids_m, ids1.to(torch.int64)) and torch.equal(sc_m, s1.double())
        one = ShardedCosineIndex(docs, 0, row_group=rg, n_groups=G)
        i2, s2 = one.rerank_groups(qs, cand, k)
        assert torch.equal(i2, ids1.to(torch.int64)) and torch.equal(s2, s1.double())
    bad = cand.copy()
    bad[3, 5] = G                                                    # owned by no shard
    with pytest.raises(ValueError):
        ShardedCosineIndex(docs, 0, row_group=rg, n_groups=G).rerank_groups(qs, bad, 10)
    bad[3, 5] = -2
    with pytest.raises(ValueError):
        ShardedCosineIndex(docs, 0, row_group=rg, n_groups=G).rerank_groups(qs, bad, 10)


# ------------------------------------------------------------------------------------------------ 7. bad input
def _status(ix, qs, cand, k, d=None, n_groups=None, null_queries=False):
    """The C call's own status for an index's tensors (d / n_groups overridable)."""
    from document_retrieval_b200 import _lib
    lib = _lib.load()
    q = None if null_queries else qs.to(ix.device, torch.bfloat16).contiguous()
    cd = None if cand is None else torch.as_tensor(cand).to(ix.device, torch.int32).contiguous()
    nq = 0 if q is None else q.shape[0]
    ids = None if nq == 0 else torch.empty((nq, max(k, 1)), dtype=torch.int32, device=ix.device)
    sims = None if nq == 0 else torch.empty((nq, max(k, 1)), dtype=torch.float32, device=ix.device)
    c = 1 if cd is None else cd.shape[1]
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    return lib.br_cosine_rerank_grouped(p(ix.docs), p(ix.inv_norm), ix.n_docs, ix.dim if d is None else d, p(ix.row_group),
                                        ix.n_groups if n_groups is None else n_groups, p(q), nq, p(cd), c, k, p(ids),
                                        p(sims), _lib.stream_ptr(ix.device))


@gpu
def test_bad_input():
    from document_retrieval_b200._lib import BRError
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator().manual_seed(71)
    docs = torch.randn(3000, 64, generator=g).to(torch.bfloat16)
    qs = torch.randn(9, 64, generator=g).to(torch.bfloat16)
    rg = np.repeat(np.arange(300), 10)
    cand = np.tile(np.arange(0, 300, 7), (9, 1))
    dec = rg.copy()
    dec[1500], dec[1501] = dec[1501], dec[1500] - 1                   # decreasing at 1501
    assert _status(CosineIndex(docs, row_group=dec), qs, cand, 10) == BR_ERR_INVALID
    assert _status(CosineIndex(docs, row_group=rg, n_groups=299), qs, cand[:, :40], 10) == BR_ERR_INVALID   # value >= n_groups
    with pytest.raises(BRError):
        CosineIndex(docs, row_group=dec).rerank_groups(qs, cand, 10)
    ix = CosineIndex(docs, row_group=rg, n_groups=310)
    for v in (-2, 310):
        c2 = cand.copy()
        c2[4, 3] = v
        assert _status(ix, qs, c2, 10) == BR_ERR_INVALID
        with pytest.raises(BRError):
            ix.rerank_groups(qs, c2, 10)
    for k in (0, 1025):
        assert _status(ix, qs, cand, k) == BR_ERR_INVALID
    assert _status(ix, qs[:, :60], cand, 10, d=60) == BR_ERR_UNSUPPORTED                 # d % 8 != 0
    wide = CosineIndex(torch.randn(500, 1032, generator=g).to(torch.bfloat16), row_group=np.repeat(np.arange(50), 10))
    assert _status(wide, torch.randn(3, 1032, generator=g), np.tile(np.arange(50), (3, 1)), 10) == BR_ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        CosineIndex(docs).rerank_groups(qs, cand, 10)
    assert _status(ix, qs, None, 10, null_queries=True) == 0         # nq = 0 with NULL pointers
    ids, sims = ix.rerank_groups(qs, cand, 10)                       # the index still answers correctly
    ref_ids, ref_sims, gs = rerank_grouped_np(docs.float().numpy(), qs.float().numpy(), rg, 310, cand, 10)
    _check(ids.cpu().numpy(), sims.cpu().numpy(), ref_ids, ref_sims, gs, np.arange(310) < 300)
    assert torch.equal(ids, _via_rows(ix, qs, cand, 10)[0])


# ------------------------------------------------------------------------------------------------ CPU
def test_restatement_matches_a_plain_loop():
    rng = np.random.default_rng(81)
    sizes = np.r_[0, rng.integers(0, 6, 40), 0, 0]
    rg = np.repeat(np.arange(sizes.size), sizes)
    docs = rng.standard_normal((rg.size, 16)).astype(np.float32)
    docs[5:9] = docs[4]                                               # exact ties across rows
    qs = np.r_[docs[4:5], rng.standard_normal((6, 16)).astype(np.float32)]
    cand = rng.integers(-1, sizes.size, (qs.shape[0], 30))
    cand[:, 10:15] = cand[:, :5]                                      # repeats
    ids, val, _ = rerank_grouped_np(docs, qs, rg, sizes.size, cand, 12)
    dn = docs / (np.linalg.norm(docs, axis=1, keepdims=True) + np.float32(1e-10))
    qn = qs / (np.linalg.norm(qs, axis=1, keepdims=True) + np.float32(1e-10))
    s = qn @ dn.T
    for i in range(qs.shape[0]):
        best = {}
        for r, gid in enumerate(rg):
            if gid in set(cand[i].tolist()):
                best[gid] = max(best.get(gid, -np.inf), s[i, r])
        want = sorted(best, key=lambda x: (-best[x], x))[:12]
        assert ids[i, :len(want)].tolist() == want and (ids[i, len(want):] == -1).all()
        np.testing.assert_allclose(val[i, :len(want)], [best[x] for x in want], rtol=1e-6)


def test_local_group_candidates():
    from document_retrieval_b200.sharded import local_group_candidates
    cand = np.array([[-1, 0, 4, 5, 9, 10, 5]])
    loc, n = local_group_candidates(cand, 5, 5)
    assert loc.tolist() == [[-1, -1, -1, 0, 4, -1, 0]] and n == 3 and loc.dtype == torch.int32
