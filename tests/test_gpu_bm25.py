"""GPU parity tests (B200): the CUDA path through the C ABI against the oracle and the golden
fixtures made from the unmodified reference.  Bar: top-k doc ids bit-exact (ties by doc id),
float64 top-k scores equal to the oracle's, dense fp32 scores within 1e-5 relative."""
import io
import pickle

import numpy as np
import pytest
import torch

from oracle import bm25_oracle as orc
from oracle.c_oracle import COracle
from document_retrieval_b200 import synth

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5   # north_star: BM25 scores within 1e-5 relative in fp32


def _q(g, i):
    return g["q_terms"][int(g["q_offsets"][i]):int(g["q_offsets"][i + 1])]


def _model(g, **kw):
    from document_retrieval_b200 import BM25
    return BM25.from_token_ids(g["doc_offsets"], g["token_ids"], int(g["vocab"]), **kw)


def _assert_dense_close(got, want):
    scale = np.maximum(np.abs(want), np.abs(want).max() * 1e-3 + 1e-30)
    assert np.max(np.abs(got - want) / scale) < REL_TOL


def test_library_loaded_and_version():
    from document_retrieval_b200 import _lib
    assert b"sm_100a" in _lib.load().br_version()


@pytest.mark.parametrize("name", ["nb_small", "nb_c1slice"])
def test_index_build_matches_oracle_and_reference(golden, name):
    g = golden(name)
    m = _model(g)
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    c = m._export_csr()
    assert np.array_equal(c["row_ptr"], ix.row_ptr) and np.array_equal(c["doc"], ix.post_doc)
    assert np.array_equal(c["tf"], ix.post_tf) and np.array_equal(c["dl"], ix.dl)
    df, idf = m._export_df_idf()
    assert np.array_equal(df, g["df"])
    assert np.array_equal(idf[df > 0], g["idf"][df > 0])            # bit-exact vs math.log of the reference
    assert m.avgdl == float(g["avgdl"]) and m.corpus_size == int(g["corpus_size"])


@pytest.mark.parametrize("name", ["nb_small", "nb_c1slice"])
def test_topk_matches_reference_golden(golden, name):
    g = golden(name)
    m = _model(g)
    ids, sc = m.retrieve_top_n_batch((g["q_terms"], g["q_offsets"]), 10)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    assert np.array_equal(ids, g["top_ids"])
    np.testing.assert_allclose(sc, g["top_scores"], rtol=1e-13, atol=0)
    # and bit-equal to the oracle (same ascending-term summation order)
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    for i in range(0, g["q_offsets"].size - 1, 7):
        oi, os_ = orc.topk_canonical(orc.get_scores(ix, _q(g, i)), 10)
        assert np.array_equal(oi, ids[i]) and np.array_equal(os_, sc[i])


def test_dense_scores_match_reference_golden(golden):
    g = golden("nb_small")
    m = _model(g)
    got = m.get_scores_batch((g["q_terms"], g["q_offsets"])).double().cpu().numpy()
    _assert_dense_close(got, g["scores"])
    one = m.get_scores(_q(g, 0))
    assert one.dtype == np.float64 and one.shape == (m.corpus_size,)
    _assert_dense_close(one, g["scores"][0])


def test_full_ranking_and_single_query_api(golden):
    g = golden("nb_small")
    m = _model(g)
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    for i in range(3):
        s = orc.get_scores(ix, _q(g, i))
        full = m.retrieve_top_n(_q(g, i), n=m.corpus_size + 5)              # n >= N, :208-209
        assert full.size == m.corpus_size and np.array_equal(full, orc.topk_canonical(s, m.corpus_size)[0])
        assert np.array_equal(m.retrieve_top_n(_q(g, i), 10), g["top_ids"][i])
        assert np.array_equal(m.get_top_n(_q(g, i), 3), g["top_ids"][i][:3])
        ex = m.exact_scores(_q(g, i)).cpu().numpy()
        assert np.array_equal(ex, s)                                          # float64 bit-exact


def test_edge_cases(golden):
    g = golden("edge_small")
    m = _model(g)
    got = m.get_scores_batch((g["q_terms"], g["q_offsets"])).double().cpu().numpy()
    _assert_dense_close(got, g["scores"])
    ids, sc = m.retrieve_top_n_batch((g["q_terms"], g["q_offsets"]), 4)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    for i in range(g["q_offsets"].size - 1):
        oi = np.lexsort((np.arange(8), -g["scores"][i]))[:4]
        assert np.array_equal(ids[i], oi), (i, ids[i], oi)
    assert ids[1].tolist()[:3] == [0, 1, 5]          # exact ties -> doc id order
    assert ids[3].tolist() == [0, 1, 2, 3] and not sc[3].any()   # OOV-only query: zeros in doc order
    # empty batch entries and an empty query
    ids2, _ = m.retrieve_top_n_batch([[], [0], []], 2)
    assert ids2.cpu().numpy()[0].tolist() == [0, 1]


def test_okapi_top100_matches_team_run1_golden(golden):
    g, t = golden("nb_small"), golden("team_run1_top100")
    m = _model(g, variant="okapi", dedup_query=False)
    ids, sc, cnt = m.retrieve_top_n_batch((g["q_terms"], g["q_offsets"]), 100, positive_only=True, return_counts=True)
    ids, sc, cnt = ids.cpu().numpy(), sc.cpu().numpy(), cnt.cpu().numpy()
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    assert np.array_equal(cnt, t["cnt"])
    for i in range(cnt.size):
        oi, os_ = orc.score_documents_for_query(ix, _q(g, i))
        n = cnt[i]
        assert np.array_equal(ids[i, :n], oi) and np.array_equal(sc[i, :n], os_)
        assert (ids[i, n:] == -1).all()
        s = orc.get_scores(ix, _q(g, i), "okapi", dedup=False)
        assert np.array_equal(s[ids[i, :n]], s[t["top"][i, :n]])     # same score sequence as heapq.nlargest


@pytest.mark.parametrize("variant,dedup", [("notebook", True), ("okapi", False), ("okapi_no_plus1", True)])
def test_c1_full_vs_c_oracle(variant, dedup):
    c = synth.make_config("C1")
    from document_retrieval_b200 import BM25
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], variant=variant, dedup_query=dedup)
    co = COracle(c["doc_offsets"], c["token_ids"], c["vocab"], variant=variant)
    pos = variant == "okapi"
    oi, os_, oc = co.topk_batch(c["q_terms"], c["q_offsets"], 10, dedup=dedup, positive_only=pos)
    ids, sc, cnt = m.retrieve_top_n_batch((c["q_terms"], c["q_offsets"]), 10, positive_only=pos, return_counts=True)
    assert np.array_equal(ids.cpu().numpy(), oi)
    assert np.array_equal(sc.cpu().numpy(), os_)
    assert np.array_equal(cnt.cpu().numpy(), oc)
    rec = np.mean([c["qrels"][i] in oi[i] for i in range(oi.shape[0])])
    if variant != "okapi_no_plus1":          # negative idf (df > N/2) legitimately hurts recall
        assert rec > 0.9
    st = m.query_stats()
    assert st["kernel_launches"] > 0 and st["postings_bytes"] > 0


def test_large_k_and_k_ge_hits():
    c = synth.make_config("C1", scale=0.2)
    from document_retrieval_b200 import BM25
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    co = COracle(c["doc_offsets"], c["token_ids"], c["vocab"])
    for k in (1, 100, 1000):
        oi, os_, _ = co.topk_batch(c["q_terms"], c["q_offsets"], k)
        ids, sc = m.retrieve_top_n_batch((c["q_terms"], c["q_offsets"]), k)
        assert np.array_equal(ids.cpu().numpy(), oi) and np.array_equal(sc.cpu().numpy(), os_)


def test_string_api_and_attributes(golden):
    g = golden("nb_small")
    from document_retrieval_b200 import BM25
    docs = synth.to_strings(g["doc_offsets"], g["token_ids"])
    qs = synth.queries_to_strings(g["q_offsets"], g["q_terms"], int(g["vocab"]))
    m = BM25(docs, k1=1.5, b=0.75)
    assert m.corpus_size == len(docs) and m.avgdl == float(g["avgdl"])
    for i in (0, 5, 40, 41, 42):
        assert np.array_equal(m.retrieve_top_n(qs[i], n=10), g["top_ids"][i])
    df, idf = m.df, m.idf
    t0 = docs[0][0]
    tid = int(t0[1:])
    assert df[t0] == g["df"][tid] and idf[t0] == g["idf"][tid]
    assert m.inverted_index[t0] == sorted(set(d for d in range(len(docs)) if t0 in docs[d]))
    assert m.term_freqs[0][t0] == docs[0].count(t0)
    assert m.doc_lengths[3] == len(docs[3])
    with pytest.raises(ZeroDivisionError):
        BM25([])


def test_pickle_roundtrip(golden):
    g = golden("nb_small")
    from document_retrieval_b200 import BM25
    docs = synth.to_strings(g["doc_offsets"], g["token_ids"])
    m = BM25(docs)
    buf = io.BytesIO()
    pickle.dump(m, buf)                       # joblib.dump(bm25_model, ...) uses pickle underneath
    m2 = pickle.loads(buf.getvalue())
    qs = synth.queries_to_strings(g["q_offsets"], g["q_terms"], int(g["vocab"]))
    for i in (0, 7, 21):
        assert np.array_equal(m2.retrieve_top_n(qs[i], n=10), g["top_ids"][i])


def test_recall_and_routing(golden):
    from document_retrieval_b200 import BM25, evaluate_recall_at_k, retrieve_test_queries, retrieve_top_n_batch
    langs, queries = synth.make_c2(scale=0.01)
    models, maps, oracles = {}, {}, {}
    for lang, c in langs.items():
        if lang == "ko":
            continue                                            # an unknown language must be skipped
        models[lang] = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
        maps[lang] = [f"{lang}-{i}" for i in range(c["n_docs"])]
        oracles[lang] = orc.build_index(c["doc_offsets"], c["token_ids"], c["vocab"])
    rows = [dict(query=q["terms"], lang=q["lang"], positive_docs=f"{q['lang']}-{q['qrel']}", query_id=i)
            for i, q in enumerate(queries)]
    want_lists = []
    for r in rows:
        if r["lang"] not in models:
            want_lists.append(None)
            continue
        ids, _ = orc.retrieve_top_n(oracles[r["lang"]], r["query"], 10)
        want_lists.append([maps[r["lang"]][i] for i in ids])
    want = orc.recall_at_k(want_lists, [r["positive_docs"] for r in rows])
    got = evaluate_recall_at_k(models, maps, rows, k=10)
    assert got == want and 0 < got < 1.0001
    lists = retrieve_test_queries(models, maps, rows, k=10)
    assert lists == [w if w is not None else [] for w in want_lists]
    any_lang = next(iter(models))
    some = [r["query"] for r in rows if r["lang"] == any_lang][:3]
    out = retrieve_top_n_batch((models[any_lang], some, 10))
    assert [o.tolist() for o in out] == [orc.retrieve_top_n(oracles[any_lang], q, 10)[0].tolist() for q in some]


@pytest.mark.parametrize("k", [3, 5, 10, 16, 32])
def test_fused_path_equals_dense_path(k):
    """The tiled smem-accumulator path and the dense path must return identical ids / scores, for k across the k <= 32
    path (threshold seeding at k, in-kernel k-th lane bound, first-launch size TILE_CAP / (24 k))."""
    c = synth.make_config("C1")
    from document_retrieval_b200 import BM25
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    q = (c["q_terms"], c["q_offsets"])
    m.set_option("fused", 0)
    ids_d, sc_d = m.retrieve_top_n_batch(q, k)
    assert m.query_stats()["queries_fused"] == 0
    m.set_option("fused", 1)
    ids_f, sc_f = m.retrieve_top_n_batch(q, k)
    st = m.query_stats()
    assert st["queries_fused"] > 0.9 * c["q_offsets"].size
    assert torch.equal(ids_d, ids_f) and torch.equal(sc_d, sc_f)
    # the tile kernel makes exactly the launches br_tile_launch_count announces (a doc-sharded caller sizes its threshold
    # exchange by it): a batch of short queries served wholly by the regular fused pass, counted on its second call
    from document_retrieval_b200 import _lib
    short = [i for i in range(c["q_offsets"].size - 1) if np.unique(_q(c, i)).size <= 20][:500]
    qs = (np.concatenate([_q(c, i) for i in short]), np.concatenate([[0], np.cumsum([_q(c, i).size for i in short])]))
    m.set_option("fused_long", 0)
    for kk in (k, 100):
        m.retrieve_top_n_batch(qs, kk)
        m.retrieve_top_n_batch(qs, kk)
        st = m.query_stats()
        assert st["queries_fused"] == len(short) and st["queries_dense"] == 0
        assert st["score_launches"] == _lib.load().br_tile_launch_count(m._h, kk) >= 1
    m.set_option("fused_long", 1)
    # okapi / duplicates counted / only docs with a hit
    m2 = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], variant="okapi", dedup_query=False)
    a = m2.retrieve_top_n_batch(q, k, positive_only=True, return_counts=True)
    m2.set_option("fused", 0)
    b = m2.retrieve_top_n_batch(q, k, positive_only=True, return_counts=True)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_fused_path_single_query_and_small_batches():
    c = synth.make_config("C1", scale=0.3)
    from document_retrieval_b200 import BM25
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"])
    co = COracle(c["doc_offsets"], c["token_ids"], c["vocab"])
    oi, os_, _ = co.topk_batch(c["q_terms"], c["q_offsets"], 10)
    for i in (0, 1, 17):
        q = c["q_terms"][c["q_offsets"][i]:c["q_offsets"][i + 1]]
        assert np.array_equal(m.retrieve_top_n(q, 10), oi[i])
    for nq in (2, 3, 5):
        ids, sc = m.retrieve_top_n_batch((c["q_terms"][:c["q_offsets"][nq]], c["q_offsets"][:nq + 1]), 10)
        assert np.array_equal(ids.cpu().numpy(), oi[:nq]) and np.array_equal(sc.cpu().numpy(), os_[:nq])


def test_rerank_v3_and_tfidf_pipeline_match_reference_golden(golden, tmp_path):
    """bm25_score + rank_documents_with_cosine_similarity_and_bm25 against the fixture made from the
    unmodified reference (cosine_similarity_bm25_reranking.py:129-238)."""
    import pandas as pd
    from document_retrieval_b200 import (bm25_score, compute_idf, compute_tf_df_and_avgdl,
                                         rank_documents_with_cosine_similarity_and_bm25)
    g, r = golden("nb_small"), golden("rerank_v3")
    vocab = int(g["vocab"])
    docs = synth.to_strings(g["doc_offsets"], g["token_ids"])
    qs = synth.queries_to_strings(g["q_offsets"], g["q_terms"], vocab)
    corpus = pd.DataFrame({"docid": [f"d{i}" for i in range(len(docs))], "preprocessed_text": [" ".join(d) for d in docs]})
    queries = pd.DataFrame({"id": list(range(len(qs))), "preprocessed_query": [" ".join(q) for q in qs]})
    path = str(tmp_path) + "/"
    tf_dict, df_dict, avgdl, num_docs, model = compute_tf_df_and_avgdl(corpus, path, return_model=True)
    import os
    assert sorted(os.listdir(tmp_path)) == ["avgdl.pkl", "df_dict.pkl", "num_docs.pkl", "tf_dict.pkl"]
    assert avgdl == float(r["avgdl"]) and num_docs == int(r["num_docs"])
    for w, v in df_dict.items():
        assert v == r["df"][int(w[1:])]
    assert tf_dict[docs[0][0]]["d0"] == docs[0].count(docs[0][0])
    idf_dict = compute_idf(df_dict, num_docs)
    for w, v in list(idf_dict.items())[:50]:
        assert v == r["idf"][int(w[1:])]                       # np.log, same ufunc as the reference
    # bm25_score on explicit pairs (batched through the same kernel)
    nq = len(qs)
    got = model.rerank_scores_v3(qs, r["pair_docs"].astype(np.int32)).cpu().numpy()
    np.testing.assert_allclose(got, r["pair_scores"], rtol=1e-12, atol=1e-15)
    one = bm25_score(qs[0], f"d{int(r['pair_docs'][0, 0])}", tf_dict, idf_dict, avgdl)
    np.testing.assert_allclose(one, r["pair_scores"][0, 0], rtol=1e-12, atol=1e-15)
    # full pipeline: compare the ranks whose order is defined in the reference (strictly positive,
    # pairwise distinct re-rank scores; the rest depends on argsort's order among equal cosines)
    ranked = rank_documents_with_cosine_similarity_and_bm25(corpus, queries, tf_dict, idf_dict, avgdl, batch_size=16)
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], vocab)
    checked = 0
    for i in range(nq):
        ref = [int(d) for d in r["top10"][i] if d >= 0]
        mine = [int(d[1:]) for d in ranked[i]]
        sc = [orc.bm25_score_rerank(ix, g["q_terms"][g["q_offsets"][i]:g["q_offsets"][i + 1]], d, r["idf"], float(r["avgdl"]))
              for d in ref]
        for j, d in enumerate(ref):
            well_defined = sc[j] > 1e-9 and all(abs(sc[j] - s2) > 1e-9 * abs(sc[j]) for jj, s2 in enumerate(sc) if jj != j)
            if not well_defined:
                break
            assert mine[j] == d, (i, j, mine, ref)
            checked += 1
    assert checked > 50


def test_long_and_duplicate_heavy_queries():
    """Queries with more than 32 terms (dense path, wider fp32 band) and heavy duplication."""
    c = synth.make_config("C1", scale=0.3)
    from document_retrieval_b200 import BM25
    rng = np.random.default_rng(11)
    qs = []
    for i in range(12):
        d = int(rng.integers(0, c["n_docs"]))
        toks = c["token_ids"][c["doc_offsets"][d]:c["doc_offsets"][d + 1]]
        qs.append(np.concatenate([toks[:60], toks[:5], toks[:5]]).astype(np.int32))   # ~50 distinct terms, duplicates
    q_off = np.cumsum([0] + [q.size for q in qs]).astype(np.int32)
    q_terms = np.concatenate(qs)
    for variant, dedup in (("notebook", True), ("okapi", False)):
        m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], variant=variant, dedup_query=dedup)
        co = COracle(c["doc_offsets"], c["token_ids"], c["vocab"], variant=variant)
        oi, os_, _ = co.topk_batch(q_terms, q_off, 10, dedup=dedup)
        ids, sc = m.retrieve_top_n_batch((q_terms, q_off), 10)
        assert np.array_equal(ids.cpu().numpy(), oi) and np.array_equal(sc.cpu().numpy(), os_)
        assert m.query_stats()["queries_dense"] == len(qs)
        # the same batch through the C entry point with n_terms an upper bound of q_offsets[nq]: the redo pass reads
        # back only the batch's own terms (q_terms is the head of a larger buffer)
        from document_retrieval_b200 import _lib
        from document_retrieval_b200._lib import ptr
        buf = torch.full((q_terms.size + 4096,), 7, dtype=torch.int32, device="cuda")
        buf[:q_terms.size] = torch.from_numpy(q_terms).cuda()
        d_off = torch.from_numpy(q_off).cuda()
        ids_c = torch.empty_like(ids)
        sc_c = torch.empty_like(sc)
        _lib.check(_lib.load().br_topk_batch(m._h, ptr(buf), ptr(d_off), len(qs), buf.numel(), 10, int(dedup), 0, ptr(ids_c),
                                             ptr(sc_c), None, _lib.stream_ptr(ids.device)), "br_topk_batch")
        torch.cuda.synchronize()
        assert torch.equal(ids_c, ids) and torch.equal(sc_c, sc) and m.query_stats()["queries_dense"] == len(qs)
        # 33..64 term occurrences (a 17-token query with its bigrams is 33 terms, bm25_ranking.ipynb:105-107): the
        # long-query pass of the tiled scorer, nothing left for the dense path
        mid = [np.concatenate([q[:36], q[:4]]) for q in qs] + [q[:33] for q in qs]
        mo = np.cumsum([0] + [q.size for q in mid]).astype(np.int32)
        mt = np.concatenate(mid)
        oi2, os2, _ = co.topk_batch(mt, mo, 10, dedup=dedup)
        ids2, sc2 = m.retrieve_top_n_batch((mt, mo), 10)
        assert np.array_equal(ids2.cpu().numpy(), oi2) and np.array_equal(sc2.cpu().numpy(), os2)
        st = m.query_stats()
        assert st["queries_dense"] == 0 and st["queries_fused"] == len(mid), st
        m.set_option("fused_long", 0)
        ids3, sc3 = m.retrieve_top_n_batch((mt, mo), 10)
        assert torch.equal(ids3, ids2) and torch.equal(sc3, sc2) and m.query_stats()["queries_dense"] == len(mid)


@pytest.mark.parametrize("k", [33, 100, 257, 1024])
def test_large_k_fused_path_equals_dense_path(k):
    """32 < k <= 1024 runs through the tiled path too (radix-select tighten over 8192-slot candidate regions) and must
    return exactly what the dense radix-select path returns - ids, float64 scores and counts."""
    c = synth.make_config("C1")
    from document_retrieval_b200 import BM25
    q = (c["q_terms"], c["q_offsets"])
    for kw, call in (({}, {}), ({"variant": "okapi", "dedup_query": False}, {"positive_only": True})):
        m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], **kw)
        a = m.retrieve_top_n_batch(q, k, return_counts=True, **call)
        assert m.query_stats()["queries_fused"] > 0.8 * (c["q_offsets"].size - 1)
        m.set_option("fused", 0)
        b = m.retrieve_top_n_batch(q, k, return_counts=True, **call)
        assert m.query_stats()["queries_fused"] == 0
        assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("k", [10, 100, 1000])
def test_massive_ties_fall_back_exactly(k):
    """20k identical docs: every score ties, the candidate band holds the whole corpus, the tiled path overflows its
    candidate regions and must hand the query to the dense path - the answer is the first k doc ids."""
    from document_retrieval_b200 import BM25
    n = 20_000
    off = np.arange(n + 1, dtype=np.int64) * 3
    tok = np.tile(np.asarray([0, 1, 2], np.int32), n)
    m = BM25.from_token_ids(off, tok, 4)
    q = (np.asarray([0, 2, 0, 3, 1], np.int32), np.asarray([0, 2, 4, 5], np.int32))     # [0,2], [0,3(df=0)], [1]
    ids, sc = m.retrieve_top_n_batch(q, k)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    for i in range(3):
        assert np.array_equal(ids[i], np.arange(k)), (i, ids[i][:12])
        assert np.all(sc[i] == sc[i][0]) and sc[i][0] > 0
    # a second corpus where only every 7th doc matches: ties among the matching docs, zeros after them
    tok2 = tok.copy().reshape(n, 3)
    tok2[np.arange(n) % 7 != 0] = [1, 1, 2]
    m2 = BM25.from_token_ids(off, tok2.reshape(-1), 4)
    ids2, sc2 = m2.retrieve_top_n_batch((np.asarray([0], np.int32), np.asarray([0, 1], np.int32)), k)
    want = np.arange(0, n, 7)[:k]
    assert np.array_equal(ids2.cpu().numpy()[0][:want.size], want)


def test_tfidf_candidate_stage_is_exact(golden):
    """a11: the TF-IDF cosine stage returns the reference's top-200 candidate SET (float64 cosine, band + re-score)
    and its cosines, cosine_similarity_bm25_reranking.py:210-229.  The query norm is a float32 BLAS dot in the
    reference (platform-dependent last bit), hence 3e-7 on the values and on what counts as a tie at the cut."""
    from document_retrieval_b200 import BM25
    g, r = golden("nb_small"), golden("rerank_v3")
    m = BM25.from_token_ids(g["doc_offsets"], g["token_ids"], int(g["vocab"]), variant="okapi_no_plus1", dedup_query=False)
    ids, sc = m.tfidf_cosine_top_n_batch((g["q_terms"], g["q_offsets"]), 200)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    nq = g["q_offsets"].size - 1
    checked = 0
    for i in range(nq):
        cos = r["cos_all"][i]
        srt = np.sort(cos)[::-1]
        np.testing.assert_allclose(sc[i], cos[ids[i]], rtol=3e-7, atol=1e-12)
        assert np.all(np.diff(sc[i]) <= 0)
        if srt[199] - srt[200] > 3e-7 * max(srt[199], 1e-30):
            assert set(ids[i].tolist()) == set(r["cos_top200"][i].tolist()), i
            checked += 1
        else:                                          # tie at the cut (zero cosines): everything strictly above it must be in
            must = set(np.flatnonzero(cos > srt[199] * (1 + 3e-7)).tolist())
            assert must <= set(ids[i].tolist())
    assert checked >= 35


def test_tfidf_stage_tiled_path_equals_dense_path():
    """The TF-IDF candidate stage runs on the tiled scorer (weight table tf*idf^2/||d||, no deferral, k = 200 -> large-k
    candidate regions, float64 re-score of the band); it must return exactly what the dense scatter-add path returns."""
    from document_retrieval_b200 import BM25
    c = synth.make_config("C1")
    q = (c["q_terms"], c["q_offsets"])
    nq = c["q_offsets"].size - 1
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], variant="okapi_no_plus1", dedup_query=False)
    for k in (10, 200):
        m.set_option("fused", 1)
        a = m.tfidf_cosine_top_n_batch(q, k)
        assert m.query_stats()["queries_fused"] > 0.8 * nq
        m.set_option("fused", 0)
        b = m.tfidf_cosine_top_n_batch(q, k)
        assert m.query_stats()["queries_fused"] == 0
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_language_filtered_pipeline_and_per_language_recall(golden):
    """text_preprocessing_and_embedding_setup.py:333-352,534-562: candidates restricted to the query's language
    (per-language GPU sub-indexes finalised with the global statistics) against the numpy restatement."""
    import pandas as pd
    from document_retrieval_b200 import (compute_idf, compute_tf_df_and_avgdl, per_language_recall,
                                         rank_documents_with_cosine_similarity_and_bm25_lang)
    g, r = golden("nb_small"), golden("rerank_v3")
    vocab = int(g["vocab"])
    docs = synth.to_strings(g["doc_offsets"], g["token_ids"])
    qs = synth.queries_to_strings(g["q_offsets"], g["q_terms"], vocab)
    langs = ["en", "fr", "de"]
    doc_lang = {f"d{i}": langs[i % 3] for i in range(len(docs))}
    corpus = pd.DataFrame({"docid": [f"d{i}" for i in range(len(docs))], "preprocessed_text": [" ".join(d) for d in docs]})
    ql = [langs[i % 3] if i % 7 else "xx" for i in range(len(qs))]          # "xx": a language without docs
    queries = pd.DataFrame({"id": list(range(len(qs))), "preprocessed_query": [" ".join(q) for q in qs], "lang": ql})
    tf_dict, df_dict, avgdl, num_docs = compute_tf_df_and_avgdl(corpus)
    idf_dict = compute_idf(df_dict, num_docs)
    ranked, qlang = rank_documents_with_cosine_similarity_and_bm25_lang(corpus, queries, tf_dict, idf_dict, avgdl, doc_lang,
                                                                        batch_size=16, n_candidates=40, k=10)
    assert qlang == dict(enumerate(ql))
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], vocab)
    lang_arr = np.array([doc_lang[f"d{i}"] for i in range(len(docs))])
    q_ids = [g["q_terms"][g["q_offsets"][i]:g["q_offsets"][i + 1]] for i in range(len(qs))]
    want = orc.rank_cosine_then_bm25(ix, q_ids, r["idf"], float(r["avgdl"]), n_candidates=40, k=10, doc_lang=lang_arr, query_lang=ql)
    checked = 0
    for i in range(len(qs)):
        mine = [int(d[1:]) for d in ranked[i]]
        if ql[i] == "xx":
            assert mine == []
            continue
        assert all(lang_arr[d] == ql[i] for d in mine)
        ref_ids, cand, cos = want[i]
        if cos.size == 40 and cos[-1] > 0:             # cut not inside the zero-cosine tail
            sc = [orc.bm25_score_rerank(ix, q_ids[i], int(d), r["idf"], float(r["avgdl"])) for d in ref_ids]
            if all(abs(a - b) > 1e-9 * max(abs(a), 1e-30) for a, b in zip(sc[:-1], sc[1:])):
                assert mine == ref_ids.tolist(), i
                checked += 1
    assert checked >= 15
    pos = [f"d{int(x)}" for x in g["qrels"]] + ["d0"] * (len(qs) - g["qrels"].size)
    got = per_language_recall(ranked, pos, qlang)
    exp = orc.per_language_recall([ranked[i] for i in range(len(qs))], pos, ql)
    assert got == exp
