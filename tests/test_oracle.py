"""CPU: pin the oracle restatements (numpy + plain C) against the golden fixtures made from the
unmodified reference (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from oracle import bm25_oracle as orc
from oracle.c_oracle import COracle
from document_retrieval_b200 import synth


def _q(g, i):
    return g["q_terms"][int(g["q_offsets"][i]):int(g["q_offsets"][i + 1])]


@pytest.mark.parametrize("name", ["nb_small", "nb_c1slice"])
def test_numpy_oracle_matches_reference_notebook(golden, name):
    g = golden(name)
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    assert ix.avgdl == float(g["avgdl"]) and ix.n_docs == int(g["corpus_size"])
    assert np.array_equal(ix.df, g["df"])
    idf = orc.idf_table(ix.df, ix.n_docs, "notebook")
    assert np.array_equal(np.isnan(idf), np.isnan(g["idf"]))
    assert np.array_equal(idf[ix.df > 0], g["idf"][ix.df > 0])          # bit-exact math.log
    nq = g["q_offsets"].size - 1
    for i in range(nq):
        s = orc.get_scores(ix, _q(g, i))
        ids, sc = orc.topk_canonical(s, 10)
        assert np.array_equal(ids, g["top_ids"][i])
        np.testing.assert_allclose(sc, g["top_scores"][i], rtol=1e-13, atol=0)
        if "scores" in g:
            np.testing.assert_allclose(s, g["scores"][i], rtol=1e-13, atol=0)
    for i in range(3):  # n >= N: full ranking (bm25_ranking.ipynb:208-209)
        s = orc.get_scores(ix, _q(g, i))
        ids, _ = orc.topk_canonical(s, ix.n_docs + 5)
        assert ids.size == ix.n_docs
        assert np.array_equal(s[ids], s[g["full_rank"][i]])


@pytest.mark.parametrize("name", ["nb_small", "nb_c1slice"])
def test_c_oracle_matches_numpy_and_golden(golden, name):
    g = golden(name)
    co = COracle(g["doc_offsets"], g["token_ids"], int(g["vocab"]), variant="notebook", n_threads=2)
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    e = co.export()
    assert np.array_equal(e["row_ptr"], ix.row_ptr) and np.array_equal(e["doc"], ix.post_doc)
    assert np.array_equal(e["tf"], ix.post_tf) and np.array_equal(e["df"], g["df"])
    assert np.array_equal(e["idf"][ix.df > 0], g["idf"][ix.df > 0])
    ids, sc, cnt = co.topk_batch(g["q_terms"], g["q_offsets"], 10)
    assert np.array_equal(ids, g["top_ids"]) and (cnt == 10).all()
    np.testing.assert_allclose(sc, g["top_scores"], rtol=1e-13, atol=0)
    for i in range(5):
        assert np.array_equal(co.get_scores(_q(g, i)), orc.get_scores(ix, _q(g, i)))


def test_edge_cases(golden):
    g = golden("edge_small")
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    co = COracle(g["doc_offsets"], g["token_ids"], int(g["vocab"]), n_threads=1)
    for i in range(g["q_offsets"].size - 1):
        s = orc.get_scores(ix, _q(g, i))
        np.testing.assert_allclose(s, g["scores"][i], rtol=1e-13, atol=0)
        assert np.array_equal(s, co.get_scores(_q(g, i)))
    # exact ties resolve by doc id: docs 0,1,5 are identical
    ids, sc = orc.topk_canonical(orc.get_scores(ix, _q(g, 1)), 3)
    assert sc[0] == sc[1] == sc[2] and ids.tolist() == [0, 1, 5]
    # OOV-only query: all zeros -> lowest doc ids
    ids, sc = orc.topk_canonical(orc.get_scores(ix, _q(g, 3)), 4)
    assert ids.tolist() == [0, 1, 2, 3] and not sc.any()


def test_team_run1_top100(golden):
    g, t = golden("nb_small"), golden("team_run1_top100")
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    co = COracle(g["doc_offsets"], g["token_ids"], int(g["vocab"]), variant="okapi", n_threads=2)
    cids, _, ccnt = co.topk_batch(g["q_terms"], g["q_offsets"], 100, dedup=False, positive_only=True)
    for i in range(g["q_offsets"].size - 1):
        ids, sc = orc.score_documents_for_query(ix, _q(g, i))
        n = int(t["cnt"][i])
        assert ids.size == n == ccnt[i]
        ref = t["top"][i, :n]
        s = orc.get_scores(ix, _q(g, i), "okapi", dedup=False)
        # heapq.nlargest is stable (first-seen wins among equal scores); canonical order is by id
        assert np.array_equal(s[ids], s[ref])
        assert sorted(ids.tolist()) == sorted(ref.tolist()) or s[ids[-1]] == s[ref[-1]]
        assert np.array_equal(cids[i, :n], ids)


def test_rerank_v3(golden):
    g, r = golden("nb_small"), golden("rerank_v3")
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    assert np.array_equal(ix.df, r["df"]) and ix.avgdl == float(r["avgdl"])
    idf = orc.idf_table(ix.df, ix.n_docs, "okapi_no_plus1")
    np.testing.assert_allclose(idf[ix.df > 0], r["idf"][ix.df > 0], rtol=1e-15)   # np.log vs math.log
    for i in range(g["q_offsets"].size - 1):
        for j in range(8):
            got = orc.bm25_score_rerank(ix, _q(g, i), int(r["pair_docs"][i, j]), r["idf"], float(r["avgdl"]))
            np.testing.assert_allclose(got, r["pair_scores"][i, j], rtol=1e-13, atol=0)


def test_tfidf_cosine_pipeline(golden):
    """cosine_similarity_bm25_reranking.py:198-238 restated (tfidf_cosine_scores / rank_cosine_then_bm25) against the
    reference's own float64 cosine matrix, its top-200 candidates and its final top-10."""
    g, r = golden("nb_small"), golden("rerank_v3")
    ix = orc.build_index(g["doc_offsets"], g["token_ids"], int(g["vocab"]))
    nq = g["q_offsets"].size - 1
    qs = [_q(g, i) for i in range(nq)]
    for i in range(nq):
        np.testing.assert_allclose(orc.tfidf_cosine_scores(ix, qs[i], r["idf"]), r["cos_all"][i], rtol=0, atol=2e-15)
    res = orc.rank_cosine_then_bm25(ix, qs, r["idf"], float(r["avgdl"]), n_candidates=200, k=10)
    defined = 0
    for i in range(nq):
        srt = np.sort(r["cos_all"][i])[::-1]
        if srt[199] > srt[200]:                       # the reference's own cut is not inside a tie
            assert set(res[i][1].tolist()) == set(r["cos_top200"][i].tolist())
            defined += 1
        if srt[9] > 0:
            assert res[i][0].tolist() == [int(d) for d in r["top10"][i] if d >= 0]
    assert defined >= 35
    # language filter: restricting the order to one language == ranking that language's docs alone
    lang = np.arange(ix.n_docs) % 3
    ql = [i % 3 for i in range(nq)]
    fl = orc.rank_cosine_then_bm25(ix, qs, r["idf"], float(r["avgdl"]), n_candidates=50, k=10, doc_lang=lang, query_lang=ql)
    for i in range(nq):
        assert all(lang[d] == ql[i] for d in fl[i][1])
        cos = r["cos_all"][i]
        mine = np.flatnonzero(lang == ql[i])
        want = mine[np.lexsort((mine, -cos[mine]))][:50]
        assert fl[i][1].tolist() == want.tolist()
    overall, per = orc.per_language_recall([[1, 2], [3], [4]], [2, 9, 4], ["en", "en", "fr"])
    assert overall == 2 / 3 and per == {"en": 0.5, "fr": 1.0}


def test_cosine_oracle(golden):
    import torch
    g = golden("cosine_small")
    d = torch.from_numpy(g["docs_bf16"]).view(torch.bfloat16).float().numpy()
    q = torch.from_numpy(g["queries_bf16"]).view(torch.bfloat16).float().numpy()
    ids, sims = orc.cosine_topk(d, q, 10)
    assert np.array_equal(ids, g["top_ids"])
    np.testing.assert_allclose(sims, g["top_sims"], rtol=1e-5, atol=1e-7)


def test_synth_deterministic():
    a = synth.make_config("C1", scale=0.1)
    b = synth.make_config("C1", scale=0.1)
    assert np.array_equal(a["token_ids"], b["token_ids"]) and np.array_equal(a["q_terms"], b["q_terms"])
    assert a["token_ids"].max() < a["vocab"] and (a["q_terms"] == a["vocab"]).sum() >= 1  # OOV present

