"""Appending documents to an index: the index of A with B appended (br_index_append, then br_index_finalize) must equal
the index of A + B built from scratch bit for bit - CSR, df, idf, statistics - and so return the same ids, float64
scores and counts from every query path.  Each test first checks that the case it was designed for happened."""
import pickle
import struct

import numpy as np
import pytest
import torch

from document_retrieval_b200 import BM25, _lib, synth
from document_retrieval_b200._lib import BRError
from document_retrieval_b200.ingest import Vocabulary
from test_gpu_handles import _assert_cycles_return_memory

pytestmark = pytest.mark.gpu

BR_ERR_STATE = -3
VARIANTS = ["notebook", "okapi", "okapi_no_plus1"]


def _parts(do, tk, cuts):
    """(doc_offsets, token_ids) of the docs [cuts[i], cuts[i+1]) of a corpus, offsets rebased to 0."""
    out = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        out.append((do[a:b + 1] - do[a], tk[do[a]:do[b]]))
    return out


def _grow(parts, vocab, **kw):
    """Index of parts[0], then every other part appended; the vocabulary grows to what each prefix needs, then to vocab."""
    seen = 0
    m = None
    for i, (o, t) in enumerate(parts):
        seen = max(seen, int(t.max()) + 1 if t.size else 1)
        v = vocab if i == len(parts) - 1 else seen
        if m is None:
            m = BM25.from_token_ids(o, t, v, **kw)
        else:
            m.add_token_ids(o, t, v)
    return m


def _queries(do, tk, vocab, nq=300, key=5):
    q_off, q_terms, _ = synth.make_queries(do, tk, nq, vocab, key=(key,))
    return q_terms, q_off


def assert_same_index(a, b):
    ca, cb = a._export_csr(), b._export_csr()
    for k in ("row_ptr", "doc", "tf", "dl"):
        np.testing.assert_array_equal(ca[k], cb[k], err_msg=k)
    (dfa, idfa), (dfb, idfb) = a._export_df_idf(), b._export_df_idf()
    np.testing.assert_array_equal(dfa, dfb)
    assert np.array_equal(idfa.view(np.int64), idfb.view(np.int64))          # NaN where df == 0 included
    assert a.stats() == b.stats()
    assert struct.pack("<d", a.avgdl) == struct.pack("<d", b.avgdl)
    assert (a.corpus_size, a.vocab_size) == (b.corpus_size, b.vocab_size)


def assert_same_topk(a, b, q, ks=(1, 10, 100, 1000)):
    for dedup in (True, False):
        a.dedup_query = b.dedup_query = dedup
        for k in ks:
            for pos in (False, True):
                ra = a.retrieve_top_n_batch(q, k, positive_only=pos, return_counts=True)
                rb = b.retrieve_top_n_batch(q, k, positive_only=pos, return_counts=True)
                for x, y in zip(ra, rb):
                    assert torch.equal(x, y), (dedup, k, pos)


@pytest.fixture(scope="module")
def corpus():
    do, tk = synth.make_corpus(12_000, 30_000, 100, key=(71,))
    return do, tk, 30_500                                              # ids 30_000 .. 30_499 unused: A + B needs no more


@pytest.mark.parametrize("variant", VARIANTS)
def test_append_equals_rebuild_on_every_query_path(corpus, variant):
    do, tk, vocab = corpus
    parts = _parts(do, tk, [0, 9_000, 12_000])
    assert int(parts[0][1].max()) + 1 < vocab                          # the append grows the vocabulary
    ref = BM25.from_token_ids(do, tk, vocab, variant=variant)
    m = _grow(parts, vocab, variant=variant)
    assert_same_index(m, ref)
    q = _queries(do, tk, vocab)
    assert_same_topk(m, ref, q)
    if variant != "okapi_no_plus1":                                   # okapi_no_plus1 is served by the dense path only
        m.retrieve_top_n_batch(q, 10)
        assert m.query_stats()["queries_fused"] > 0
    for x in (m, ref):
        x.set_option("fused", 0)
    assert_same_topk(m, ref, q, ks=(10, 1000))
    assert m.query_stats()["queries_fused"] == 0
    for x in (m, ref):
        x.set_option("fused", 1)
    assert torch.equal(m.retrieve_records_batch(q, 50), ref.retrieve_records_batch(q, 50))
    g = torch.Generator().manual_seed(3)
    allow = torch.rand(2, ref.corpus_size, generator=g) < 0.3
    rows = torch.randint(-1, 2, (q[1].size - 1,), generator=g)
    for n in (10, 100):
        fa = m.retrieve_top_n_batch(q, n, doc_filter=allow, query_filter=rows, return_counts=True)
        fb = ref.retrieve_top_n_batch(q, n, doc_filter=allow, query_filter=rows, return_counts=True)
        assert all(torch.equal(x, y) for x, y in zip(fa, fb))
    q0 = q[0][q[1][0]:q[1][1]]
    assert torch.equal(m.exact_scores(q0), ref.exact_scores(q0))
    # fp32 scores: a one-term query adds exactly one posting weight to each doc, so the weights themselves must match bit
    # for bit; longer queries add their terms' weights with atomics in no fixed order, so they match up to fp32 rounding
    one = np.unique(q[0][q[0] < vocab])[:500].astype(np.int32)
    q1 = (one, np.arange(one.size + 1, dtype=np.int32))
    assert torch.equal(m.get_scores_batch(q1), ref.get_scores_batch(q1))
    assert torch.allclose(m.get_scores_batch(q), ref.get_scores_batch(q), rtol=1e-5, atol=1e-4)
    if variant == "okapi_no_plus1":
        # the doc norms of the TF-IDF table are float64 sums in atomic order: the cosines match to the last bits only
        ia, sa = m.tfidf_cosine_top_n_batch(q, 200)
        ib, sb = ref.tfidf_cosine_top_n_batch(q, 200)
        assert torch.equal(ia, ib) and torch.allclose(sa, sb, rtol=1e-12, atol=0)
        assert torch.equal(m.rerank_scores_v3(q, ia), ref.rerank_scores_v3(q, ib))


@pytest.mark.parametrize("n_old,n_new", [(2047, 2048), (2048, 2049), (2047, 4097), (4095, 4096), (4096, 4097),
                                         (4096, 8193), (1, 2), (3000, 3001)])
def test_append_at_sub_range_and_padding_edges(n_old, n_new):
    # sub-ranges of 2048 docs (skip tables, tile kernel) and n_pad, a multiple of 4096 (dense rows); single-doc appends
    do, tk = synth.make_corpus(n_new, 5_000, 40, key=(72, n_old))
    parts = _parts(do, tk, [0, n_old, n_new])
    ref = BM25.from_token_ids(do, tk, 5_000)
    m = _grow(parts, 5_000)
    assert m.corpus_size == n_new and parts[1][0].size - 1 == n_new - n_old
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, 5_000, nq=100), ks=(1, 10, 100))


def test_append_of_empty_docs():
    do, tk = synth.make_corpus(3_000, 5_000, 40, key=(73,))
    lens = np.diff(do)
    lens[2_500::7] = 0                                                 # docs of length 0, some of them appended
    lens[-1] = 0
    do = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    tk = tk[:do[-1]]
    ref = BM25.from_token_ids(do, tk, 5_000)
    m = _grow(_parts(do, tk, [0, 2_500, 2_999, 3_000]), 5_000)       # the last part is one empty doc
    assert m._export_csr()["dl"][-1] == 0
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, 5_000, nq=100), ks=(10, 1000))


def _with_term_in_docs(do, tk, term, docs):
    """The corpus with one more token `term` at the end of each doc in `docs`."""
    lens = np.diff(do)
    add = np.zeros_like(lens)
    add[docs] = 1
    out_off = np.concatenate([[0], np.cumsum(lens + add)]).astype(np.int64)
    out = np.empty(out_off[-1], np.int32)
    for d in range(lens.size):
        out[out_off[d]:out_off[d] + lens[d]] = tk[do[d]:do[d + 1]]
        if add[d]:
            out[out_off[d + 1] - 1] = term
    return out_off, out


def test_append_that_promotes_a_term_to_every_row_class():
    """A term rare in A is in every doc of B: after the append it is hot (skip table), a look-up row (df >= N/64), a
    streamed row (df >= N/5) and one of the 32 most frequent terms, none of which it was."""
    do, tk = synth.make_corpus(9_000, 20_000, 60, key=(74,))
    a = BM25.from_token_ids(*_parts(do, tk, [0, 6_000])[0], 20_000)
    df_a = a._export_df_idf()[0]
    rare = int(np.nonzero((df_a >= 1) & (df_a < 4))[0][-1])           # in A, but below hot_min = max(4, n_sub / 4)
    do, tk = _with_term_in_docs(do, tk, rare, np.arange(6_000, 9_000))
    parts = _parts(do, tk, [0, 6_000, 9_000])
    assert rare not in np.argsort(-df_a, kind="stable")[:32]
    ref = BM25.from_token_ids(do, tk, 20_000)
    a.add_token_ids(*parts[1], 20_000)
    df = ref._export_df_idf()[0]
    assert df[rare] >= 9_000 / 5 and rare in np.argsort(-df, kind="stable")[:32]
    assert_same_index(a, ref)
    q_terms, q_off = _queries(do, tk, 20_000)
    q_terms = np.concatenate([q_terms, [rare, 1, 7], [rare]]).astype(np.int32)
    q_off = np.concatenate([q_off, [q_off[-1] + 3, q_off[-1] + 4]]).astype(np.int32)
    assert_same_topk(a, ref, (q_terms, q_off))
    a.retrieve_top_n_batch((q_terms, q_off), 10)
    assert a.query_stats()["queries_fused"] > 0


def test_append_that_turns_an_idf_negative():
    """okapi_no_plus1: the term's df crosses N/2, so its idf changes sign."""
    do, tk = synth.make_corpus(7_000, 20_000, 60, key=(75,))
    t = 3_000
    do, tk = _with_term_in_docs(do, tk, t, np.arange(3_000, 7_000))
    parts = _parts(do, tk, [0, 3_000, 7_000])
    a = BM25.from_token_ids(*parts[0], 20_000, variant="okapi_no_plus1")
    assert a._export_df_idf()[1][t] > 0
    ref = BM25.from_token_ids(do, tk, 20_000, variant="okapi_no_plus1")
    a.add_token_ids(*parts[1], 20_000)
    assert ref._export_df_idf()[1][t] < 0
    assert_same_index(a, ref)
    q_terms, q_off = _queries(do, tk, 20_000)
    q_terms = np.concatenate([q_terms, [t, 1, 2, 3], [t]]).astype(np.int32)
    q_off = np.concatenate([q_off, [q_off[-1] + 4, q_off[-1] + 5]]).astype(np.int32)
    assert_same_topk(a, ref, (q_terms, q_off))


@pytest.mark.parametrize("kind", ["old_terms", "new_terms", "both"])
def test_append_of_old_new_and_mixed_terms(kind):
    do, tk = synth.make_corpus(6_000, 8_000, 50, key=(76,))
    n_old = 4_000
    tk = tk.copy()
    v_a = int(tk[:do[n_old]].max()) + 1
    tail = tk[do[n_old]:]
    if kind == "old_terms":
        tail %= 97                                                     # B only uses terms A has
    elif kind == "new_terms":
        tail += v_a                                                    # B only uses terms A lacks
    vocab = int(tk.max()) + 1
    new = np.setdiff1d(tail, tk[:do[n_old]])
    assert (new.size == 0) if kind == "old_terms" else (new.size == np.unique(tail).size if kind == "new_terms" else
                                                        0 < new.size < np.unique(tail).size)
    ref = BM25.from_token_ids(do, tk, vocab)
    m = _grow(_parts(do, tk, [0, n_old, 6_000]), vocab)
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, vocab, nq=200), ks=(10, 100))


def test_chain_of_appends(corpus):
    do, tk, vocab = corpus
    ref = BM25.from_token_ids(do, tk, vocab, variant="okapi")
    m = _grow(_parts(do, tk, [0, 5_000, 5_001, 8_000, 12_000]), vocab, variant="okapi")
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, vocab), ks=(10, 100))


def _texts(n_docs, key, vocab=4_000):
    do, tk = synth.make_corpus(n_docs, vocab, 30, key=(key,))
    return [" ".join(d) for d in synth.to_strings(do, tk, prefix="w")]


@pytest.mark.parametrize("bigrams", [False, True])
def test_vocabulary_extension_equals_a_build_over_all_texts(bigrams):
    texts = _texts(3_000, 77)
    a, b = texts[:2_000], texts[2_000:]
    b[5] = "brand new words " + b[5] + " été"                 # terms no doc of A has
    voc, _, _ = Vocabulary.from_texts(a, bigrams=bigrams)
    n_a = len(voc)
    b_off, b_ids = voc.extend_texts(b)
    ref, ref_off, ref_ids = Vocabulary.from_texts(a + b, bigrams=bigrams)
    assert len(voc) == len(ref) > n_a
    for x, y in zip(voc._export(), ref._export()):
        np.testing.assert_array_equal(x, y)
    assert voc.terms == ref.terms
    start = int(ref_off[2_000])
    assert torch.equal(b_ids, ref_ids[start:]) and torch.equal(b_off, ref_off[2_000:] - start)
    queries = ["brand new w1 w2", "w3 unseen w1", "été words"]
    assert all(torch.equal(x, y) for x, y in zip(voc.encode_texts(queries), ref.encode_texts(queries)))


def test_add_documents_extends_terms_like_a_build():
    texts = _texts(3_000, 78)
    docs = [t.split() for t in texts]
    docs[2_500] = docs[2_500] + ["zz_new", "w1"]
    ref = BM25(docs)
    m = BM25(docs[:2_000]).add_documents(docs[2_000:2_400]).add_documents(docs[2_400:])
    assert m.terms == ref.terms and m.vocab == ref.vocab
    assert_same_index(m, ref)
    assert m.df == ref.df and m.inverted_index == ref.inverted_index
    qs = [d[:5] for d in docs[::97]]
    assert_same_topk(m, ref, qs, ks=(10,))
    with pytest.raises(ValueError):
        BM25.from_texts(texts[:10], bigrams=True).add_documents(docs[10:20])


@pytest.mark.parametrize("bigrams", [False, True])
def test_add_texts_after_load_saves_the_same_file(tmp_path, bigrams):
    texts = _texts(3_000, 79)
    texts[2_900] += " only_in_b"
    ref = BM25.from_texts(texts, bigrams=bigrams)
    BM25.from_texts(texts[:2_000], bigrams=bigrams).save(tmp_path / "a.brix")
    m = BM25.load(tmp_path / "a.brix")
    assert m.vocabulary is None
    m.add_texts(texts[2_000:2_500]).add_texts(texts[2_500:])
    assert m.terms == ref.terms
    assert_same_index(m, ref)
    m.save(tmp_path / "grown.brix")
    ref.save(tmp_path / "ref.brix")
    assert (tmp_path / "grown.brix").read_bytes() == (tmp_path / "ref.brix").read_bytes()
    qs = [" ".join(t.split()[:4]) for t in texts[::101]] + ["only_in_b w1"]
    assert all(torch.equal(x, y) for x, y in zip(m.retrieve_top_n_texts(qs, 10), ref.retrieve_top_n_texts(qs, 10)))
    # a model built from token lists gets its GPU vocabulary from its terms first
    b = BM25([t.split() for t in texts[:2_000]]).add_texts(texts[2_000:]) if not bigrams else None
    if b is not None:
        assert b.terms == ref.terms
        assert_same_index(b, ref)
    # pickling a grown model
    u = pickle.loads(pickle.dumps(m))
    assert u.terms == ref.terms and u.corpus_size == ref.corpus_size
    assert_same_index(u, ref)


def test_add_token_ids_rules(corpus):
    do, tk, vocab = corpus
    (oa, ta), (ob, tb) = _parts(do, tk, [0, 100, 200])
    m = BM25.from_token_ids(oa, ta, vocab)
    assert m.add_token_ids(np.zeros(1, np.int64), np.zeros(0, np.int32)) is m and m.corpus_size == 100   # empty: no-op
    m.add_token_ids(torch.as_tensor(ob).cuda(), torch.as_tensor(tb).cuda())          # default vocab_size: the current
    assert m.corpus_size == 200 and m.vocab_size == vocab
    s = BM25([["a", "b"], ["b", "c"]])
    with pytest.raises(ValueError):
        s.add_token_ids(np.array([0, 1]), np.array([3], np.int32), vocab_size=4)        # a term without a string


def _query_results(m, q):
    return [m.retrieve_top_n_batch(q, k, return_counts=True) for k in (10, 1000)]


def test_refused_appends_leave_the_index_unchanged(corpus):
    do, tk, vocab = corpus
    (oa, ta), (ob, tb) = _parts(do, tk, [0, 8_000, 12_000])
    m = BM25.from_token_ids(oa, ta, vocab)
    q = _queries(do, tk, vocab, nq=200)
    before = _query_results(m, q)
    csr = {k: v.copy() for k, v in m._export_csr().items()}
    bad_tok = tb.copy()
    bad_tok[17] = vocab
    bad_off = ob.copy()
    bad_off[3], bad_off[4] = bad_off[4], bad_off[3]
    heavy = (np.array([0, 65_536], np.int64), np.full(65_536, 11, np.int32))
    cases = [(ob, bad_tok, vocab), (ob, tb, vocab - 1), (bad_off, tb, vocab), (heavy[0], heavy[1], vocab)]
    assert bad_off[3] > bad_off[4]
    lib = _lib.load()
    for o, t, v in cases:
        with pytest.raises(BRError):
            m._append_ids(o, t, v)
        assert m.corpus_size == 8_000 and m.stats()["n_docs"] == 8_000
        after = _query_results(m, q)
        assert all(torch.equal(x, y) for r0, r1 in zip(before, after) for x, y in zip(r0, r1))
        m._csr = None
        assert all(np.array_equal(csr[k], m._export_csr()[k]) for k in csr)
    m.add_token_ids(ob, tb)
    assert_same_index(m, BM25.from_token_ids(do, tk, vocab))
    # between br_index_append and br_index_finalize no query is answered
    h = BM25.from_token_ids(oa, ta, vocab)
    dev = torch.device("cuda", torch.cuda.current_device())
    d_off, d_tok = torch.as_tensor(ob, device=dev), torch.as_tensor(tb, device=dev)
    assert lib.br_index_append(h._h, d_tok.data_ptr(), d_off.data_ptr(), ob.size - 1, vocab, _lib.stream_ptr(dev)) == 0
    qt, qo = (torch.as_tensor(x, device=dev) for x in q)
    ids = torch.empty((qo.numel() - 1, 10), dtype=torch.int32, device=dev)
    sc = torch.empty((qo.numel() - 1, 10), dtype=torch.float64, device=dev)
    assert lib.br_topk_batch(h._h, qt.data_ptr(), qo.data_ptr(), qo.numel() - 1, qt.numel(), 10, 1, 0, ids.data_ptr(),
                             sc.data_ptr(), None, _lib.stream_ptr(dev)) == BR_ERR_STATE
    h.corpus_size = 12_000
    h.finalize()
    ref = BM25.from_token_ids(do, tk, vocab)
    assert torch.equal(h.retrieve_top_n_batch(q, 10)[0], ref.retrieve_top_n_batch(q, 10)[0])


def test_refused_add_texts_takes_its_terms_back():
    texts = _texts(500, 80)
    m = BM25.from_texts(texts[:400])
    n_terms = len(m.terms)
    with pytest.raises(BRError):
        m.add_texts(texts[400:] + [" ".join(["boom"] * 65_536)])     # a term 65536 times in one doc
    assert len(m.vocabulary) == n_terms and m.corpus_size == 400
    m.add_texts(texts[400:])
    ref = BM25.from_texts(texts)
    assert m.terms == ref.terms
    assert_same_index(m, ref)


def test_doc_shard_refuses_to_grow(corpus):
    do, tk, vocab = corpus
    (oa, ta), (ob, tb) = _parts(do, tk, [0, 6_000, 12_000])
    shard = BM25.from_token_ids(oa, ta, vocab, finalize=False)
    other = BM25.from_token_ids(ob, tb, vocab, finalize=False)
    df = shard.local_df_tensor().cpu().numpy().astype(np.int64) + other.local_df_tensor().cpu().numpy()
    shard.finalize(12_000, shard.stats()["sum_dl"] + other.stats()["sum_dl"], df)
    with pytest.raises(BRError):
        shard.add_token_ids(ob, tb)
    s2 = BM25([["a", "b"], ["b"]])
    s2.finalize(10, 30, np.array([5, 7]))
    with pytest.raises(BRError):
        s2.add_documents([["a"]])
    with pytest.raises(BRError):
        s2.add_texts(["a b"])
    assert shard.corpus_size == 6_000 and s2.corpus_size == 2


def test_append_cycles_return_memory(corpus):
    do, tk, vocab = corpus
    parts = _parts(do, tk, [0, 10_000, 12_000])

    def cycle():
        m = _grow(parts, vocab)
        assert m.corpus_size == 12_000
        m.retrieve_top_n_batch([[1, 2, 3]], 10)
        del m

    _assert_cycles_return_memory(cycle)
