"""GPU: filtered top-k (br_topk_batch_filtered, br_topk_batch_records_filtered, br_cosine_topk_filtered).

The contract: a filtered query's result is the unfiltered call's result on the corpus restricted to the docs its filter
row allows - doc ids, N, avgdl, df and idf unchanged, so the float64 scores are bit-identical to the unfiltered ones; order
(score desc, doc id asc); positive_only=0 fills the tail with allowed zero-score docs in doc-id order; -1 pads when
fewer than k docs are allowed; row -1 = unfiltered; an all-ones row = the unfiltered call."""
import numpy as np
import pytest
import torch
from hypothesis import HealthCheck, given, settings, strategies as st

from oracle import bm25_oracle as orc
from document_retrieval_b200 import synth

pytestmark = pytest.mark.gpu
RTOL, ATOL = 1e-5, 2e-6          # cosine tolerances of test_gpu_cosine.py


def restricted_topk(scores, allowed, k, positive_only=False):
    """Canonical top-k of the corpus restricted to the allowed docs, padded to k: (ids int64 (-1 pads), scores, count)."""
    docs = np.nonzero(allowed)[0]
    li, ls = orc.topk_canonical(scores[docs], k, positive_only)
    ids = np.full(k, -1, np.int64)
    sc = np.zeros(k, np.float64)
    ids[:li.size] = docs[li]
    sc[:li.size] = ls
    return ids, sc, li.size


def pack(queries):
    q_off = np.zeros(len(queries) + 1, np.int32)
    np.cumsum([len(q) for q in queries], out=q_off[1:])
    q_terms = np.asarray([t for q in queries for t in q], np.int32)
    return q_terms, q_off


# ------------------------------------------------------------------------------------------------ 1. tiny corpora
@st.composite
def filtered_case(draw):
    vocab = draw(st.integers(1, 12))
    n_docs = draw(st.integers(1, 70))
    term = st.integers(0, vocab - 1)
    docs = draw(st.lists(st.lists(term, min_size=0, max_size=8), min_size=n_docs, max_size=n_docs))
    if not any(docs):
        docs[0] = [0]
    queries = draw(st.lists(st.lists(st.integers(-1, vocab + 2), min_size=0, max_size=10), min_size=1, max_size=6))
    k = draw(st.integers(1, n_docs))
    rows = []
    for _ in range(draw(st.integers(1, 4))):
        kind = draw(st.sampled_from(["empty", "ones", "one", "random", "few"]))
        if kind == "empty":
            r = np.zeros(n_docs, bool)
        elif kind == "ones":
            r = np.ones(n_docs, bool)
        elif kind == "one":
            r = np.zeros(n_docs, bool)
            r[draw(st.integers(0, n_docs - 1))] = True
        elif kind == "random":
            r = np.asarray(draw(st.lists(st.booleans(), min_size=n_docs, max_size=n_docs)), bool)
        else:                                                   # fewer allowed docs than k
            r = np.zeros(n_docs, bool)
            r[draw(st.lists(st.integers(0, n_docs - 1), max_size=max(0, k - 1)))] = True
        rows.append(r)
    qrow = draw(st.lists(st.integers(-1, len(rows) - 1), min_size=len(queries), max_size=len(queries)))
    variant = draw(st.sampled_from(["notebook", "okapi", "okapi_no_plus1"]))
    return vocab, docs, queries, k, np.stack(rows), np.asarray(qrow, np.int32), variant, draw(st.booleans()), draw(st.booleans())


@settings(max_examples=150, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
@given(filtered_case())
def test_filtered_topk_equals_oracle_on_tiny_corpora(case):
    from document_retrieval_b200 import BM25
    vocab, docs, queries, k, rows, qrow, variant, dedup, positive_only = case
    off = np.zeros(len(docs) + 1, np.int64)
    np.cumsum([len(d) for d in docs], out=off[1:])
    tok = np.asarray([t for d in docs for t in d], np.int32)
    ix = orc.build_index(off, tok, vocab)
    m = BM25.from_token_ids(off, tok, vocab, variant=variant, dedup_query=dedup)
    q = pack(queries)
    ids, sc, cnt = m.retrieve_top_n_batch(q, k, positive_only=positive_only, return_counts=True, doc_filter=rows,
                                          query_filter=qrow)
    ids, sc, cnt = ids.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    u_ids, u_sc, u_cnt = (x.cpu().numpy() for x in m.retrieve_top_n_batch(q, k, positive_only=positive_only,
                                                                          return_counts=True))
    for i, qt in enumerate(queries):
        allowed = np.ones(len(docs), bool) if qrow[i] < 0 else rows[qrow[i]]
        oi, os_, oc = restricted_topk(orc.get_scores(ix, qt, variant, dedup), allowed, k, positive_only)
        assert np.array_equal(ids[i], oi), (case, i, ids[i], oi)
        assert np.array_equal(sc[i], os_), (case, i, sc[i], os_)
        assert cnt[i] == oc, (case, i, cnt[i], oc)
        if allowed.all():                                       # all-ones row / row -1: the unfiltered call, bit for bit
            assert np.array_equal(ids[i], u_ids[i]) and np.array_equal(sc[i], u_sc[i]) and cnt[i] == u_cnt[i]
    # one [N] filter for the whole batch, and the records entry point
    ids1, sc1 = m.retrieve_top_n_batch(q, k, positive_only=positive_only, doc_filter=rows[0])
    rec = m.retrieve_records_batch(q, k, positive_only=positive_only, doc_filter=rows[0]).cpu()
    assert np.array_equal(rec[..., 0].numpy(), ids1.cpu().numpy().astype(np.int64))
    assert np.array_equal(rec[..., 1].contiguous().view(torch.float64).numpy(), sc1.cpu().numpy())
    for i, qt in enumerate(queries):
        oi, os_, _ = restricted_topk(orc.get_scores(ix, qt, variant, dedup), rows[0], k, positive_only)
        assert np.array_equal(ids1[i].cpu().numpy(), oi) and np.array_equal(sc1[i].cpu().numpy(), os_)
    # single-query surface, including the n >= N full ranking
    got = m.retrieve_top_n(np.asarray(queries[0], np.int32), len(docs) + 2, doc_filter=rows[0])
    full_i, _, c = restricted_topk(orc.get_scores(ix, queries[0], variant, dedup), rows[0], len(docs))
    assert np.array_equal(got, full_i[:c])


# ------------------------------------------------------------------------------------------------ 2. C4-shaped slice
N_C4 = 1_000_000


@pytest.fixture(scope="module")
def c4_filtered():
    from oracle.c_oracle import COracle
    from document_retrieval_b200 import BM25
    do, tk = synth.make_corpus_torch(N_C4, N_C4, 60, "cuda", seed=5)
    qo, qt, _ = synth.make_queries_torch(do, tk, 600, N_C4, seed=6)
    queries = [qt[qo[i]:qo[i + 1]] for i in range(qo.size - 1)]
    # long queries: > 32 terms (long tiled pass) and > 64 terms (dense path), e.g. bigram-expanded text
    queries += [np.concatenate(queries[i:i + 4]) for i in range(0, 40, 4)]
    queries += [np.concatenate(queries[i:i + 8]) for i in range(40, 120, 8)]
    assert max(len(x) for x in queries) > 64 and sum(32 < len(x) <= 64 for x in queries) >= 5
    q = pack(queries)
    rng = np.random.Generator(np.random.PCG64(77))
    rows = np.stack([rng.random(N_C4) < 0.5, rng.random(N_C4) < 0.05, rng.random(N_C4) < 0.001,
                     np.zeros(N_C4, bool)])
    rows[3, 250_000:350_000] = True                              # a contiguous range
    qrow = (np.arange(len(queries)) % 6 - 1).astype(np.int32)    # -1 (unfiltered) and rows 0..3, 4 wraps to row 0
    qrow[qrow == 4] = 0
    co = COracle(do.cpu().numpy(), tk.cpu().numpy(), N_C4)
    want = {10: [], 100: []}
    for i, x in enumerate(queries):
        s = co.get_scores(x)
        allowed = np.ones(N_C4, bool) if qrow[i] < 0 else rows[qrow[i]]
        for kk in want:
            want[kk].append(restricted_topk(s, allowed, kk))
    return BM25.from_token_ids(do, tk, N_C4), q, rows, qrow, want


@pytest.mark.parametrize("k", [10, 100])
@pytest.mark.parametrize("opt", [("defer_pm", 0), ("defer_pm", 1000), ("fused", 0), ("fused_long", 0)])
def test_c4_slice_filtered_against_the_oracle(c4_filtered, k, opt):
    m, q, rows, qrow, want = c4_filtered
    defaults = {"defer_pm": 650, "fused": 1, "fused_long": 1}
    m.set_option(*opt)
    try:
        ids, sc, cnt = m.retrieve_top_n_batch(q, k, return_counts=True, doc_filter=rows, query_filter=qrow)
        st_ = m.query_stats()
    finally:
        m.set_option(opt[0], defaults[opt[0]])
    if opt[0] != "fused":
        assert st_["queries_fused"] > 0 and st_["queries_dense"] > 0     # the dense fallback sees a filtered sub-batch
    ids, sc, cnt = ids.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    for i, (oi, os_, oc) in enumerate(want[k]):
        assert np.array_equal(ids[i], oi), (opt, k, i)
        assert np.array_equal(sc[i], os_), (opt, k, i)
        assert cnt[i] == oc, (opt, k, i)


# ------------------------------------------------------------------------------------------------ 3. language rows
def test_language_rows_equal_per_language_subindexes():
    """One index over a multi-language corpus + one filter row per language == the per-language sub-indexes finalised
    with the global statistics (functional._lang_models_for), mapped to global ids - bit for bit."""
    from document_retrieval_b200 import BM25
    n, vocab, n_lang = 200_000, 200_000, 7
    do, tk = synth.make_corpus_torch(n, vocab, 60, "cuda", seed=41)
    qo, qt, _ = synth.make_queries_torch(do, tk, 350, vocab, seed=42)
    lang = np.random.Generator(np.random.PCG64(43)).integers(0, n_lang, n)
    full = BM25.from_token_ids(do, tk, vocab)
    st_ = full.stats()
    df = full.local_df_tensor().to(torch.int64).cpu().numpy()
    rows = np.stack([lang == l for l in range(n_lang)])
    qlang = (np.arange(qo.size - 1) % n_lang).astype(np.int32)
    do_c, tk_c = do.cpu().numpy(), tk.cpu().numpy()
    for k in (10, 1000):
        ids, sc = full.retrieve_top_n_batch((qt, qo), k, doc_filter=rows, query_filter=qlang)
        ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
        for l in range(n_lang):
            docs = np.nonzero(lang == l)[0]
            if k == 10 or l == 0:
                lens = do_c[docs + 1] - do_c[docs]
                off = np.zeros(docs.size + 1, np.int64)
                np.cumsum(lens, out=off[1:])
                toks = np.concatenate([tk_c[do_c[d]:do_c[d + 1]] for d in docs])
                sub = BM25.from_token_ids(off, toks, vocab, finalize=False)
                sub.finalize(st_["n_docs"], st_["sum_dl"], df)
                assert sub.avgdl == full.avgdl
            qs = np.nonzero(qlang == l)[0]
            if k == 1000 and l != 0:
                continue                                            # k = 1000: one language (many large-k launches)
            sq = pack([qt[qo[i]:qo[i + 1]] for i in qs])
            si, ss = sub.retrieve_top_n_batch(sq, k)
            si, ss = si.cpu().numpy(), ss.cpu().numpy()
            mapped = np.where(si >= 0, docs[np.maximum(si, 0)], -1)
            assert np.array_equal(ids[qs], mapped), (k, l)
            assert np.array_equal(sc[qs], ss), (k, l)


# ------------------------------------------------------------------------------------------------ 4. sharded BM25
def _shards(c, world):
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.sharded import shard_bounds
    shards = []
    for lo, hi in shard_bounds(c["n_docs"], world):
        do = c["doc_offsets"][lo:hi + 1] - c["doc_offsets"][lo]
        tk = c["token_ids"][c["doc_offsets"][lo]:c["doc_offsets"][hi]]
        shards.append(BM25.from_token_ids(do, tk, c["vocab"], doc_base=lo, finalize=False))
    df = sum(s.local_df_tensor().to(torch.int64) for s in shards).cpu().numpy()
    n_stat = sum(s.stats()["n_docs"] for s in shards)
    sum_dl = sum(s.stats()["sum_dl"] for s in shards)
    for s in shards:
        s.finalize(n_stat, sum_dl, df)
    return shards


def _filter_rows(n, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    rows = np.stack([rng.random(n) < 0.3, rng.random(n) < 0.01, np.zeros(n, bool)])
    rows[2, [3, n // 2, n - 5]] = True                             # 3 allowed docs: fewer than k
    return rows


@pytest.mark.parametrize("world", [2, 3])
def test_fake_shards_filtered_equal_single_index(world):
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.sharded import local_filter_slice, merge_topk_cuda
    c = synth.make_config("C1", scale=0.5)
    q = (c["q_terms"], c["q_offsets"])
    nq = c["q_offsets"].size - 1
    rows = _filter_rows(c["n_docs"], 5)
    qrow = (np.arange(nq) % 4 - 1).astype(np.int32)
    single = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    ids1, sc1 = single.retrieve_top_n_batch(q, 10, doc_filter=rows, query_filter=qrow)
    assert int((ids1 < 0).sum()) > 0                               # short results are part of the check
    all_ids, all_sc = [], []
    for s in _shards(c, world):
        ids, sc = s.retrieve_top_n_batch(q, 10, doc_filter=local_filter_slice(rows, s.doc_base, s.corpus_size),
                                         query_filter=qrow)
        all_ids.append(torch.where(ids >= 0, ids.to(torch.int64) + s.doc_base, torch.full_like(ids, -1, dtype=torch.int64)))
        all_sc.append(sc)
    ids_m, sc_m = merge_topk_cuda(torch.stack(all_ids), torch.stack(all_sc), 10)
    assert torch.equal(ids_m, ids1.to(torch.int64)) and torch.equal(sc_m, sc1)


def test_filtered_threshold_exchange_with_a_second_shard_equals_single_index():
    """As test_gpu_sharded's exchange test, with a filter: shard A prunes with thresholds that include shard B's
    filtered k best scores; merged with B's filtered result it equals the filtered single index bit for bit once the
    queries that come back short - fewer than min(k, allowed docs) entries: their zero-score fill needs local thresholds -
    are repeated without the exchange, as ShardedBM25 does."""
    from document_retrieval_b200 import BM25, _lib
    from document_retrieval_b200._lib import check
    from document_retrieval_b200.sharded import local_filter_slice, merge_topk_cuda
    k = 10
    c = synth.make_config("C1", scale=1.0)
    q = (c["q_terms"], c["q_offsets"])
    nq = c["q_offsets"].size - 1
    rows = _filter_rows(c["n_docs"], 6)
    qrow = (np.arange(nq) % 4 - 1).astype(np.int32)
    single = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    ids1, sc1 = single.retrieve_top_n_batch(q, k, doc_filter=rows, query_filter=qrow)
    a, b = _shards(c, 2)
    fa = local_filter_slice(rows, a.doc_base, a.corpus_size)
    fb = local_filter_slice(rows, b.doc_base, b.corpus_size)
    ids_b, sc_b = b.retrieve_top_n_batch(q, k, doc_filter=fb, query_filter=qrow)
    other = (sc_b * (1.0 - 1e-6)).to(torch.float32)
    other = torch.where(ids_b >= 0, other, torch.zeros_like(other)).contiguous()
    other_thr = torch.where(ids_b[:, k - 1] >= 0, other[:, k - 1], torch.zeros_like(other[:, 0])).contiguous()

    def wrap(p, n):
        class _Arr:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (p, False), "version": 3}
        return torch.as_tensor(_Arr(), device="cuda")

    def exchange(local_ptr, gathered_ptr, n_floats, stream, user):
        try:
            local, gathered = wrap(local_ptr, n_floats), wrap(gathered_ptr, 2 * n_floats)
            gathered[:n_floats].copy_(local)
            gathered[n_floats:].copy_((other_thr if n_floats == nq else other).flatten())
            return 0
        except Exception:
            return -1

    lib = _lib.load()
    cb = _lib.THR_EXCHANGE_FN(exchange)
    rounds = int(lib.br_tile_launch_count(a._h, k)) - 1
    check(lib.br_set_thr_exchange(a._h, cb, None, rounds, 2), "br_set_thr_exchange")
    try:
        ids_a, sc_a = a.retrieve_top_n_batch(q, k, doc_filter=fa, query_filter=qrow)
    finally:
        check(lib.br_set_thr_exchange(a._h, None, None, -1, 1), "br_set_thr_exchange")
    glob = lambda s, ids: torch.where(ids >= 0, ids.to(torch.int64) + s.doc_base, torch.full_like(ids, -1, dtype=torch.int64))
    # B ran without the exchange and zero-filled from its own docs; a shard under the exchange returns only docs with a
    # hit, so B's list enters the first merge as such
    ids_bx = torch.where(sc_b != 0, ids_b, torch.full_like(ids_b, -1))
    ids_m, sc_m = merge_topk_cuda(torch.stack([glob(a, ids_a), glob(b, ids_bx)]), torch.stack([sc_a, sc_b]), k)
    n_allowed = np.where(qrow >= 0, rows.sum(1)[np.maximum(qrow, 0)], c["n_docs"])
    need = torch.from_numpy(np.minimum(k, n_allowed)).cuda()
    last = ids_m.gather(1, (need - 1).clamp(min=0)[:, None])[:, 0]
    short = (need > 0) & (last < 0)
    ids_a0, sc_a0 = a.retrieve_top_n_batch(q, k, doc_filter=fa, query_filter=qrow)      # local thresholds only
    i2, s2 = merge_topk_cuda(torch.stack([glob(a, ids_a0), glob(b, ids_b)]), torch.stack([sc_a0, sc_b]), k)
    ids_m[short], sc_m[short] = i2[short], s2[short]
    assert torch.equal(ids_m, ids1.to(torch.int64)) and torch.equal(sc_m, sc1)


# ------------------------------------------------------------------------------------------------ 5. cosine
def _masked_ref(docs, qs, allowed, k):
    """torch fp32 reference (team_run1.py:270-282) with the disallowed rows at -inf -> (ids, sims, full scores)."""
    d = docs.float()
    dn = d / (d.norm(dim=1, keepdim=True) + 1e-10)
    qn = qs.float() / (qs.float().norm(dim=1, keepdim=True) + 1e-10)
    full = qn @ dn.T
    masked = torch.where(allowed, full, torch.full_like(full, -float("inf")))
    v, i = torch.topk(masked, k, dim=1)
    return i, v, full


def _check_cos(ids, sims, allowed, docs, qs, k):
    ref_i, ref_v, full = _masked_ref(docs, qs, allowed, k)
    ids, sims = ids.cpu(), sims.cpu()
    ref_i, ref_v, full, allowed = ref_i.cpu(), ref_v.cpu(), full.cpu(), allowed.cpu()
    n_allowed = allowed.sum(1)
    for i in range(ids.shape[0]):
        c = int(min(k, n_allowed[i]))
        assert (ids[i, c:] == -1).all() and (sims[i, c:] == 0).all()
        got = ids[i, :c]
        assert (got >= 0).all() and allowed[i, got].all()
        np.testing.assert_allclose(sims[i, :c].numpy(), ref_v[i, :c].numpy(), rtol=RTOL, atol=ATOL)
        if not torch.equal(got, ref_i[i, :c]):
            np.testing.assert_allclose(full[i, got].numpy(), ref_v[i, :c].numpy(), rtol=RTOL, atol=ATOL)
            assert len(set(got.tolist())) == c


@pytest.mark.parametrize("kernel", [0, 1])
@pytest.mark.parametrize("n,d,nq,k", [(20000, 384, 300, 10), (5000, 768, 250, 32), (3000, 1024, 200, 10)])
def test_filtered_cosine_topk(kernel, n, d, nq, k):
    from document_retrieval_b200.cosine import CosineIndex, set_cosine_option
    g = torch.Generator(device="cuda").manual_seed(synth.ROOT_SEED + n + d)
    docs = torch.randn(n, d, generator=g, device="cuda").to(torch.bfloat16)
    qs = torch.randn(nq, d, generator=g, device="cuda").to(torch.bfloat16)
    rows = torch.stack([torch.rand(n, generator=g, device="cuda") < p for p in (0.5, 0.02, 0.001)]
                       + [torch.ones(n, dtype=torch.bool, device="cuda")])
    rows[2, :] = False
    rows[2, [5, n // 3, n - 1]] = True                              # 3 allowed rows: fewer than k -> -1 padding
    qrow = (torch.arange(nq, device="cuda") % 5 - 1).to(torch.int32)
    ix = CosineIndex(docs)
    set_cosine_option("kernel", kernel)
    try:
        ids, sims = ix.topk(qs, k, doc_filter=rows, query_filter=qrow)
        ids_u, sims_u = ix.topk(qs, k)
    finally:
        set_cosine_option("kernel", 0)
    allowed = torch.where((qrow >= 0)[:, None], rows[qrow.clamp(min=0).long()], torch.ones_like(rows[:1]))
    _check_cos(ids, sims, allowed, docs, qs, k)
    unf = (qrow < 0) | (qrow == 3)                                  # row -1 and the all-ones row: the unfiltered call
    assert torch.equal(ids[unf], ids_u[unf]) and torch.equal(sims[unf], sims_u[unf])
    assert (ids[qrow == 2][:, 3:] == -1).all()


def test_filtered_cosine_overflow_fallback_with_ties():
    """Thousands of identical rows: the candidate filter overflows and the exact gather pass answers - it must give the
    redone queries only their allowed rows."""
    from document_retrieval_b200.cosine import CosineIndex
    g = torch.Generator(device="cuda").manual_seed(3)
    n, d, k = 12000, 256, 16
    docs = torch.randn(n, d, generator=g, device="cuda").to(torch.bfloat16)
    docs[2000:6000] = docs[2000]                                    # 4000 duplicates
    qs = torch.cat([docs[2000:2001], docs[2000:2001], torch.randn(30, d, generator=g, device="cuda").to(torch.bfloat16)])
    rows = torch.ones(2, n, dtype=torch.bool, device="cuda")
    rows[0, 2000:5000:2] = False                                    # every other duplicate of the first half excluded
    rows[1, 2000:5990] = False                                      # only 10 duplicates left, fewer than k
    qrow = torch.tensor([0, 1] + [0] * 30, dtype=torch.int32, device="cuda")
    ids, sims = CosineIndex(docs).topk(qs, k, doc_filter=rows, query_filter=qrow)
    want0 = torch.nonzero(rows[0, 2000:6000]).flatten()[:k] + 2000
    assert torch.equal(ids[0], want0)
    assert torch.equal(ids[1, :10], torch.arange(5990, 6000, device="cuda"))
    allowed = rows[qrow.long()]
    _check_cos(ids[2:], sims[2:], allowed[2:], docs, qs[2:], k)


def test_filtered_fake_cosine_shards_equal_single_index():
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.sharded import ShardedCosineIndex, local_filter_slice, merge_topk_cuda, shard_bounds
    g = torch.Generator(device="cuda").manual_seed(9)
    docs = torch.randn(20_000, 256, generator=g, device="cuda").to(torch.bfloat16)
    docs[777] = docs[12_345]
    qs = torch.cat([torch.randn(300, 256, generator=g, device="cuda").to(torch.bfloat16), docs[777:778]])
    rows = torch.stack([torch.rand(20_000, generator=g, device="cuda") < 0.2, torch.ones(20_000, dtype=torch.bool, device="cuda")])
    rows[0, [777, 12_345]] = True
    qrow = (torch.arange(301, device="cuda") % 3 - 1).to(torch.int32)
    ids1, s1 = CosineIndex(docs).topk(qs, 10, doc_filter=rows, query_filter=qrow)
    parts = [CosineIndex(docs[lo:hi], doc_base=lo).topk(qs, 10, doc_filter=local_filter_slice(rows, lo, hi - lo), query_filter=qrow)
             for lo, hi in shard_bounds(20_000, 3)]
    ids_m, sc_m = merge_topk_cuda(torch.stack([p[0] for p in parts]), torch.stack([p[1].double() for p in parts]), 10)
    assert torch.equal(ids_m, ids1) and torch.equal(sc_m, s1.double())
    one = ShardedCosineIndex(docs, 0)                               # one rank: the global filter is its own
    i2, s2 = one.topk(qs, 10, doc_filter=rows, query_filter=qrow)
    assert torch.equal(i2, ids1) and torch.equal(s2, s1.double())


# ------------------------------------------------------------------------------------------------ 6. errors
def test_filter_errors():
    from document_retrieval_b200 import BM25
    from document_retrieval_b200._lib import BRError
    from document_retrieval_b200.cosine import CosineIndex
    c = synth.make_config("C1", scale=0.2)
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    q = (c["q_terms"], c["q_offsets"])
    nq, n = c["q_offsets"].size - 1, c["n_docs"]
    rows = np.ones((2, n), bool)
    rows[1, ::2] = False
    bad = np.zeros(nq, np.int32)
    bad[nq // 2] = 2                                                # outside [-1, 2)
    with pytest.raises(BRError):
        m.retrieve_top_n_batch(q, 10, doc_filter=rows, query_filter=bad)
    bad[nq // 2] = -2
    with pytest.raises(BRError):
        m.retrieve_records_batch(q, 10, doc_filter=rows, query_filter=bad)
    good = (np.arange(nq) % 2).astype(np.int32)                     # the handle still answers the next batch correctly
    ids, sc = m.retrieve_top_n_batch(q, 10, doc_filter=rows, query_filter=good)
    ref = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    ids_u, sc_u = ref.retrieve_top_n_batch(q, 10)
    g0, g1 = torch.from_numpy(good == 0).cuda(), torch.from_numpy(good == 1).cuda()
    assert torch.equal(ids[g0], ids_u[g0]) and torch.equal(sc[g0], sc_u[g0])
    assert ((ids[g1] % 2 == 1) | (ids[g1] < 0)).all()
    for kw in (dict(doc_filter=rows[0][:-1]),                          # wrong N
               dict(doc_filter=rows),                                  # [F, N] without query_filter
               dict(doc_filter=rows, query_filter=good[:-1]),          # wrong Q
               dict(doc_filter=rows[0].astype(np.int32)),              # not bool
               dict(doc_filter=rows[0], query_filter=good)):           # query_filter with a 1-D filter
        with pytest.raises(ValueError):
            m.retrieve_top_n_batch(q, 10, **kw)
    docs = torch.randn(500, 64, device="cuda").to(torch.bfloat16)
    ix = CosineIndex(docs)
    qs = torch.randn(7, 64, device="cuda").to(torch.bfloat16)
    with pytest.raises(BRError):
        ix.topk(qs, 5, doc_filter=torch.ones(1, 500, dtype=torch.bool), query_filter=torch.tensor([0, 0, 0, 1, 0, 0, 0]))
    with pytest.raises(ValueError):
        ix.topk(qs, 5, doc_filter=torch.ones(499, dtype=torch.bool))
    ids, _ = ix.topk(qs, 5, doc_filter=torch.ones(500, dtype=torch.bool))
    assert torch.equal(ids, ix.topk(qs, 5)[0])
