"""Removing documents from an index: the index of C with the docs R removed (br_index_remove, then br_index_finalize) must
equal the index built from scratch from the docs of C not in R, in order, over the same vocabulary, bit for bit - CSR,
df, idf, statistics - and so return the same ids, float64 scores and counts from every query path.  Each test first
checks that the case it was designed for happened."""
import pickle

import numpy as np
import pytest
import torch

from document_retrieval_b200 import BM25, _lib, synth
from document_retrieval_b200._lib import BRError
from document_retrieval_b200.ingest import Vocabulary
from test_gpu_append import _parts, _queries, _with_term_in_docs, assert_same_index, assert_same_topk
from test_gpu_handles import _assert_cycles_return_memory

pytestmark = pytest.mark.gpu

BR_ERR_INVALID = -1
BR_ERR_STATE = -3
VARIANTS = ["notebook", "okapi", "okapi_no_plus1"]


def _kept(do, tk, remove):
    """(doc_offsets, token_ids) of the docs of a corpus whose `remove` flag is False, in order."""
    remove = np.asarray(remove, bool)
    lens = np.diff(do)
    off = np.concatenate([[0], np.cumsum(lens[~remove])]).astype(np.int64)
    return off, tk[np.repeat(~remove, lens)]


def _mask(n, ids):
    m = np.zeros(n, bool)
    m[np.asarray(ids, np.int64)] = True
    return m


def _random_mask(n, frac, key):
    return np.random.Generator(np.random.PCG64(key)).random(n) < frac


@pytest.fixture(scope="module")
def corpus():
    do, tk = synth.make_corpus(12_000, 30_000, 100, key=(81,))
    return do, tk, 30_500                                              # ids 30_000 .. 30_499 unused


@pytest.mark.parametrize("variant", VARIANTS)
def test_remove_equals_rebuild_on_every_query_path(corpus, variant):
    do, tk, vocab = corpus
    rm = _random_mask(12_000, 0.25, 82)
    m = BM25.from_token_ids(do, tk, vocab, variant=variant)
    ref = BM25.from_token_ids(*_kept(do, tk, rm), vocab, variant=variant)
    df_all, df_kept = m._export_df_idf()[0], ref._export_df_idf()[0]
    assert 2_800 < rm.sum() < 3_200 and np.any((df_all > 0) & (df_kept == 0))   # some terms lose every posting
    assert m.remove_documents(rm) is m
    assert m.corpus_size == ref.corpus_size == 12_000 - rm.sum()
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
    g = torch.Generator().manual_seed(4)
    allow = torch.rand(2, ref.corpus_size, generator=g) < 0.3        # filters of the new width
    rows = torch.randint(-1, 2, (q[1].size - 1,), generator=g)
    for n in (10, 100):
        fa = m.retrieve_top_n_batch(q, n, doc_filter=allow, query_filter=rows, return_counts=True)
        fb = ref.retrieve_top_n_batch(q, n, doc_filter=allow, query_filter=rows, return_counts=True)
        assert all(torch.equal(x, y) for x, y in zip(fa, fb))
    q0 = q[0][q[1][0]:q[1][1]]
    assert torch.equal(m.exact_scores(q0), ref.exact_scores(q0))
    # a one-term query adds exactly one posting weight to each doc: the fp32 weights themselves must match bit for bit
    one = np.unique(q[0][q[0] < vocab])[:500].astype(np.int32)
    q1 = (one, np.arange(one.size + 1, dtype=np.int32))
    assert torch.equal(m.get_scores_batch(q1), ref.get_scores_batch(q1))
    if variant == "okapi_no_plus1":
        # the doc norms of the TF-IDF table are float64 sums in atomic order: the cosines match to the last bits only
        ia, sa = m.tfidf_cosine_top_n_batch(q, 200)
        ib, sb = ref.tfidf_cosine_top_n_batch(q, 200)
        assert torch.equal(ia, ib) and torch.allclose(sa, sb, rtol=1e-12, atol=0)
        assert torch.equal(m.rerank_scores_v3(q, ia), ref.rerank_scores_v3(q, ib))


# sub-ranges of 2048 docs (skip tables, tile kernel) and n_pad, a multiple of 4096 (dense rows): N before -> N after; and
# the first doc, the last doc, one contiguous block, every other doc
EDGES = {
    "4097-first": (4097, [0]),
    "4096-last": (4096, [4095]),
    "2049-one": (2049, [1_000]),
    "8193-block": (8193, range(2_000, 6_097)),
    "2-first": (2, [0]),
    "2-last": (2, [1]),
    "6000-every-other": (6000, range(0, 6_000, 2)),
}
N_AFTER = {"4097-first": 4096, "4096-last": 4095, "2049-one": 2048, "8193-block": 4096, "2-first": 1, "2-last": 1,
           "6000-every-other": 3000}


@pytest.mark.parametrize("case", list(EDGES))
def test_remove_at_sub_range_and_padding_edges(case):
    n, ids = EDGES[case]
    do, tk = synth.make_corpus(n, 5_000, 40, key=(83, n))
    rm = _mask(n, list(ids))
    ref = BM25.from_token_ids(*_kept(do, tk, rm), 5_000)
    m = BM25.from_token_ids(do, tk, 5_000).remove_documents(np.asarray(list(ids)))
    assert m.corpus_size == ref.corpus_size == N_AFTER[case]
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, 5_000, nq=100), ks=(1, 10, 100))


def test_remove_that_demotes_a_term_from_every_row_class():
    """A term rare in the first 6 000 docs is in every doc of the block [6 000, 9 000): in the whole index it is hot (skip
    table), a look-up row (df >= N/64), a streamed row (df >= N/5) and one of the 32 most frequent terms.  Removing the
    block leaves it in none of these classes."""
    do, tk = synth.make_corpus(9_000, 20_000, 60, key=(84,))
    head = BM25.from_token_ids(*_parts(do, tk, [0, 6_000])[0], 20_000)
    df_head = head._export_df_idf()[0]
    rare = int(np.nonzero((df_head >= 1) & (df_head < 4))[0][-1])     # below hot_min = max(4, n_sub / 4)
    do, tk = _with_term_in_docs(do, tk, rare, np.arange(6_000, 9_000))
    m = BM25.from_token_ids(do, tk, 20_000)
    df = m._export_df_idf()[0]
    assert df[rare] >= 9_000 / 5 and rare in np.argsort(-df, kind="stable")[:32]
    m.remove_documents(np.arange(6_000, 9_000))
    ref = BM25.from_token_ids(*_kept(do, tk, _mask(9_000, np.arange(6_000, 9_000))), 20_000)
    df = ref._export_df_idf()[0]
    assert 1 <= df[rare] < 4 and rare not in np.argsort(-df, kind="stable")[:32]
    assert_same_index(m, ref)
    q_terms, q_off = _queries(do, tk, 20_000)
    q_terms = np.concatenate([q_terms, [rare, 1, 7], [rare]]).astype(np.int32)
    q_off = np.concatenate([q_off, [q_off[-1] + 3, q_off[-1] + 4]]).astype(np.int32)
    assert_same_topk(m, ref, (q_terms, q_off))
    m.retrieve_top_n_batch((q_terms, q_off), 10)
    assert m.query_stats()["queries_fused"] > 0


@pytest.mark.parametrize("variant", ["okapi", "okapi_no_plus1"])
def test_term_whose_every_posting_is_removed(corpus, variant):
    do, tk, vocab = corpus
    m = BM25.from_token_ids(do, tk, vocab, variant=variant)
    df = m._export_df_idf()[0]
    t = int(np.nonzero((df >= 3) & (df <= 6))[0][0])
    docs_with_t = np.unique(np.repeat(np.arange(12_000), np.diff(do))[tk == t])
    rm = _random_mask(12_000, 0.05, 85)
    rm[docs_with_t] = True
    assert docs_with_t.size == df[t]
    m.remove_documents(rm)
    ref = BM25.from_token_ids(*_kept(do, tk, rm), vocab, variant=variant)
    df2, idf2 = m._export_df_idf()
    assert df2[t] == 0 and np.isnan(idf2[t]) and t not in m.df and t not in m.idf and t not in m.inverted_index
    assert_same_index(m, ref)
    q_terms, q_off = _queries(do, tk, vocab, nq=100)
    q_terms = np.concatenate([q_terms, [t], [t, 1, 2, 3], [5, t]]).astype(np.int32)
    q_off = np.concatenate([q_off, q_off[-1] + np.array([1, 5, 7])]).astype(np.int32)
    assert_same_topk(m, ref, (q_terms, q_off))
    ids, _ = m.retrieve_top_n_batch((np.array([t], np.int32), np.array([0, 1], np.int32)), 10, positive_only=True)
    assert (ids == -1).all()                                          # no doc has the term any more


def test_remove_that_turns_an_idf_positive():
    """okapi_no_plus1: the term is in 4 000 of 7 000 docs (df > N/2, idf < 0); removing 2 000 of them leaves 2 000 of
    5 000 (idf > 0)."""
    do, tk = synth.make_corpus(7_000, 20_000, 60, key=(86,))
    t = 3_000
    do, tk = _with_term_in_docs(do, tk, t, np.arange(3_000, 7_000))
    m = BM25.from_token_ids(do, tk, 20_000, variant="okapi_no_plus1")
    assert m._export_df_idf()[1][t] < 0
    rm = _mask(7_000, np.arange(5_000, 7_000))
    m.remove_documents(rm)
    ref = BM25.from_token_ids(*_kept(do, tk, rm), 20_000, variant="okapi_no_plus1")
    assert ref._export_df_idf()[1][t] > 0
    assert_same_index(m, ref)
    q_terms, q_off = _queries(do, tk, 20_000)
    q_terms = np.concatenate([q_terms, [t, 1, 2, 3], [t]]).astype(np.int32)
    q_off = np.concatenate([q_off, [q_off[-1] + 4, q_off[-1] + 5]]).astype(np.int32)
    assert_same_topk(m, ref, (q_terms, q_off))


def test_remove_of_empty_docs():
    do, tk = synth.make_corpus(3_000, 5_000, 40, key=(87,))
    lens = np.diff(do)
    lens[::7] = 0
    do = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    tk = tk[:do[-1]]
    rm = _random_mask(3_000, 0.3, 88)
    assert ((lens == 0) & rm).any() and ((lens == 0) & ~rm).any()     # empty docs removed and kept
    m = BM25.from_token_ids(do, tk, 5_000).remove_documents(rm)
    ref = BM25.from_token_ids(*_kept(do, tk, rm), 5_000)
    assert (m._export_csr()["dl"] == 0).any()
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, 5_000, nq=100), ks=(10, 1000))


def test_remove_then_append_is_an_update(corpus):
    """The update workflow: remove the old versions, append the new ones = a build of the kept docs followed by the new."""
    do, tk, vocab = corpus
    (oa, ta), (ob, tb) = _parts(do, tk, [0, 10_000, 12_000])
    rm = _random_mask(10_000, 0.1, 89)
    m = BM25.from_token_ids(oa, ta, vocab).remove_documents(rm)
    m.add_token_ids(ob, tb)
    ka, kt = _kept(oa, ta, rm)
    ref = BM25.from_token_ids(np.concatenate([ka, ka[-1] + ob[1:]]), np.concatenate([kt, tb]), vocab)
    assert m.corpus_size == 12_000 - rm.sum()
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, vocab, nq=200), ks=(10, 100))


def test_append_then_remove(corpus):
    do, tk, vocab = corpus
    (oa, ta), (ob, tb) = _parts(do, tk, [0, 9_000, 12_000])
    rm = _random_mask(12_000, 0.2, 90)
    rm[8_990:9_010] = True                                            # across the append boundary
    m = BM25.from_token_ids(oa, ta, vocab).add_token_ids(ob, tb).remove_documents(rm)
    ref = BM25.from_token_ids(*_kept(do, tk, rm), vocab)
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, vocab, nq=200), ks=(10, 100))


def test_two_removals_equal_one_of_the_union(corpus):
    do, tk, vocab = corpus
    first = _random_mask(12_000, 0.15, 91)
    second = _random_mask(12_000, 0.15, 92) & ~first
    assert second.any()
    m = BM25.from_token_ids(do, tk, vocab, variant="okapi").remove_documents(first)
    m.remove_documents(np.nonzero(second[~first])[0])                # the second removal in the new ids
    one = BM25.from_token_ids(do, tk, vocab, variant="okapi").remove_documents(first | second)
    ref = BM25.from_token_ids(*_kept(do, tk, first | second), vocab, variant="okapi")
    assert_same_index(m, one)
    assert_same_index(m, ref)
    assert_same_topk(m, ref, _queries(do, tk, vocab, nq=200), ks=(10, 100))


def _texts(n_docs, key, vocab=4_000):
    do, tk = synth.make_corpus(n_docs, vocab, 30, key=(key,))
    return [" ".join(d) for d in synth.to_strings(do, tk, prefix="w")]


def test_token_list_model_has_the_dicts_of_the_kept_lists():
    docs = [t.split() for t in _texts(2_000, 93)]
    docs[10] = docs[10] + ["only_in_ten"]
    rm = _random_mask(2_000, 0.25, 94)
    rm[10] = True
    m = BM25(docs).remove_documents(rm)
    kept = [d for d, r in zip(docs, rm) if not r]
    ref = BM25(kept)
    assert "only_in_ten" in m.terms and "only_in_ten" not in m.df and len(m.terms) > len(ref.terms)
    assert m.df == ref.df and m.idf == ref.idf and m.inverted_index == ref.inverted_index
    assert m.term_freqs == ref.term_freqs and m.doc_lengths == ref.doc_lengths
    # BM25(kept) numbers its terms differently; the bit-exact reference is the build of the kept docs over m's term ids
    off = np.concatenate([[0], np.cumsum([len(d) for d in kept])]).astype(np.int64)
    same = BM25.from_token_ids(off, np.array([m.vocab[w] for d in kept for w in d], np.int32), m.vocab_size)
    assert_same_index(m, same)
    qs = [d[:5] for d in docs[::37]]
    q_ids = [[m.vocab[w] for w in q] for q in qs]
    assert all(torch.equal(x, y) for x, y in zip(m.retrieve_top_n_batch(qs, 10), same.retrieve_top_n_batch(q_ids, 10)))


@pytest.mark.parametrize("bigrams", [False, True])
def test_texts_model_after_removal(bigrams):
    texts = _texts(3_000, 95)
    new = _texts(200, 96)
    new[3] += " never_seen_before"
    rm = _random_mask(3_000, 0.25, 97)
    m = BM25.from_texts(texts, bigrams=bigrams)
    n_terms = len(m.vocabulary)
    m.remove_documents(rm)
    assert len(m.vocabulary) == n_terms and m.vocab_size == n_terms
    _, off, ids = Vocabulary.from_texts(texts, bigrams=bigrams)
    ref = BM25.from_token_ids(*_kept(off.cpu().numpy(), ids.cpu().numpy(), rm), n_terms)
    assert_same_index(m, ref)
    qs = [" ".join(t.split()[:4]) for t in texts[::101]] + ["w1 w2 unseen"]
    q = m.vocabulary.encode_texts(qs)
    assert all(torch.equal(x, y) for x, y in zip(m.retrieve_top_n_texts(qs, 10), ref.retrieve_top_n_batch(q, 10)))
    # a later append still extends the same vocabulary
    m.add_texts(new)
    voc, off, ids = Vocabulary.from_texts(texts + new, bigrams=bigrams)
    assert len(m.vocabulary) == len(voc) > n_terms
    ref = BM25.from_token_ids(*_kept(off.cpu().numpy(), ids.cpu().numpy(), np.concatenate([rm, np.zeros(200, bool)])),
                              len(voc))
    assert_same_index(m, ref)


def test_load_remove_save_gives_the_same_file_and_pickles(tmp_path):
    texts = _texts(3_000, 98)
    BM25.from_texts(texts).save(tmp_path / "all.brix")
    m = BM25.load(tmp_path / "all.brix")
    rm = _random_mask(3_000, 0.3, 99)
    m.remove_documents(rm)
    _, off, ids = Vocabulary.from_texts(texts)
    ref = BM25.from_token_ids(*_kept(off.cpu().numpy(), ids.cpu().numpy(), rm), m.vocab_size)
    ref.terms = list(m.terms)
    assert_same_index(m, ref)
    m.save(tmp_path / "removed.brix")
    ref.save(tmp_path / "ref.brix")
    assert (tmp_path / "removed.brix").read_bytes() == (tmp_path / "ref.brix").read_bytes()
    u = pickle.loads(pickle.dumps(m))
    assert u.terms == ref.terms and u.corpus_size == ref.corpus_size
    assert_same_index(u, ref)


def test_mask_ids_and_device_tensors_give_the_same_index(corpus):
    do, tk, vocab = corpus
    rm = _random_mask(12_000, 0.2, 100)
    ids = np.nonzero(rm)[0]
    ref = BM25.from_token_ids(*_kept(do, tk, rm), vocab)
    dup = np.concatenate([ids, ids[::3]])                              # duplicates count once
    np.random.Generator(np.random.PCG64(101)).shuffle(dup)
    forms = [rm, ids, ids.tolist(), dup, torch.as_tensor(rm).cuda(), torch.as_tensor(ids).cuda(),
             torch.as_tensor(dup.astype(np.int32)).cuda()]
    for f in forms:
        m = BM25.from_token_ids(do, tk, vocab)
        assert m.remove_documents(f) is m
        assert_same_index(m, ref)


def test_empty_removal_is_a_no_op(corpus):
    do, tk, vocab = corpus
    m = BM25.from_token_ids(do, tk, vocab)
    q = _queries(do, tk, vocab, nq=100)
    before = _query_results(m, q)
    for empty in ([], np.zeros(0, np.int64), np.zeros(12_000, bool), torch.zeros(0, dtype=torch.int64).cuda()):
        assert m.remove_documents(empty) is m and m.corpus_size == 12_000
    assert_same_index(m, BM25.from_token_ids(do, tk, vocab))
    after = _query_results(m, q)
    assert all(torch.equal(x, y) for r0, r1 in zip(before, after) for x, y in zip(r0, r1))


def _query_results(m, q):
    return [m.retrieve_top_n_batch(q, k, return_counts=True) for k in (10, 1000)]


def test_refused_removals_leave_the_index_unchanged(corpus):
    do, tk, vocab = corpus
    m = BM25.from_token_ids(do, tk, vocab)
    q = _queries(do, tk, vocab, nq=200)
    before = _query_results(m, q)
    csr = {k: v.copy() for k, v in m._export_csr().items()}

    def unchanged():
        assert m.corpus_size == 12_000 and m.stats()["n_docs"] == 12_000
        after = _query_results(m, q)
        assert all(torch.equal(x, y) for r0, r1 in zip(before, after) for x, y in zip(r0, r1))
        m._csr = None
        assert all(np.array_equal(csr[k], m._export_csr()[k]) for k in csr)

    cases = [np.array([5, 12_000]), np.array([-1, 3]), np.ones(11_999, bool), np.ones((2, 12_000), bool),
             np.array([1.0, 2.0]), torch.tensor([3.0]).cuda(), np.ones(12_000, bool), np.arange(12_000),
             torch.arange(12_000).cuda()]
    for c in cases:
        with pytest.raises(ValueError):
            m.remove_documents(c)
        unchanged()
    # through the C ABI: null pointers and a mask that removes every doc
    lib = _lib.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    st = _lib.stream_ptr(dev)
    every = torch.ones(12_000, dtype=torch.uint8, device=dev)
    assert lib.br_index_remove(m._h, every.data_ptr(), st) == BR_ERR_INVALID
    assert lib.br_index_remove(m._h, None, st) == BR_ERR_INVALID
    assert lib.br_index_remove(None, every.data_ptr(), st) == BR_ERR_INVALID
    unchanged()
    # a mask without a nonzero byte: BR_OK, and the handle still answers queries without a finalize
    assert lib.br_index_remove(m._h, torch.zeros(12_000, dtype=torch.uint8, device=dev).data_ptr(), st) == 0
    unchanged()
    # after a removal no query is answered until br_index_finalize
    rm = _random_mask(12_000, 0.2, 102)
    mask = torch.as_tensor(rm.astype(np.uint8), device=dev)
    assert lib.br_index_remove(m._h, mask.data_ptr(), st) == 0
    qt, qo = (torch.as_tensor(x, device=dev) for x in q)
    ids = torch.empty((qo.numel() - 1, 10), dtype=torch.int32, device=dev)
    sc = torch.empty((qo.numel() - 1, 10), dtype=torch.float64, device=dev)
    assert lib.br_topk_batch(m._h, qt.data_ptr(), qo.data_ptr(), qo.numel() - 1, qt.numel(), 10, 1, 0, ids.data_ptr(),
                             sc.data_ptr(), None, st) == BR_ERR_STATE
    m.corpus_size = 12_000 - int(rm.sum())
    m._csr = None
    m.finalize()
    ref = BM25.from_token_ids(*_kept(do, tk, rm), vocab)
    assert_same_index(m, ref)
    assert torch.equal(m.retrieve_top_n_batch(q, 10)[0], ref.retrieve_top_n_batch(q, 10)[0])


def test_doc_shard_refuses_removal(corpus):
    do, tk, vocab = corpus
    (oa, ta), (ob, tb) = _parts(do, tk, [0, 6_000, 12_000])
    shard = BM25.from_token_ids(oa, ta, vocab, finalize=False)
    other = BM25.from_token_ids(ob, tb, vocab, finalize=False)
    df = shard.local_df_tensor().cpu().numpy().astype(np.int64) + other.local_df_tensor().cpu().numpy()
    shard.finalize(12_000, shard.stats()["sum_dl"] + other.stats()["sum_dl"], df)
    with pytest.raises(BRError):
        shard.remove_documents([0, 5])
    assert shard.corpus_size == 6_000 and shard.stats()["n_docs"] == 6_000


def test_remove_cycles_return_memory(corpus):
    do, tk, vocab = corpus
    rm = _random_mask(12_000, 0.25, 103)

    def cycle():
        m = BM25.from_token_ids(do, tk, vocab).remove_documents(rm)
        assert m.corpus_size == 12_000 - rm.sum()
        m.retrieve_top_n_batch([[1, 2, 3]], 10)
        del m

    _assert_cycles_return_memory(cycle)
