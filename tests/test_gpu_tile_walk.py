"""GPU: the tile scorer's posting walk on slice shapes it has to get right - several slices of one sub-range packed
into one 32-posting step and straddling step boundaries, one-posting slices, sparse-class slices longer than 64
postings, dense-posting terms behind sparse ones, duplicate query terms (multiplicities) and the long-query pass.
The fused path is compared with the dense path and with the C oracle, ids and float64 scores bit for bit."""
import numpy as np
import pytest
import torch

from oracle.c_oracle import COracle

pytestmark = pytest.mark.gpu

S = 2048                      # docs per sub-range of the tile kernel (kSubShift)
N_SUB = 96
N = N_SUB * S
FILL_VOCAB = 200_000          # filler tokens: rare, routed through the cold bucket


def _designed_terms(rng):
    """term id -> doc ids.  Term classes by document frequency: hot (skip table) from n_sub / 4, dense-posting from
    N / 64 (32 per sub-range on average), streamed row from 0.2 N."""
    terms = {}
    t = 0
    for _ in range(10):           # ~10-30 postings per sub-range: slices that share and straddle 32-posting steps
        terms[t] = rng.choice(N, size=int(rng.integers(900, 2900)), replace=False); t += 1
    for _ in range(14):           # about one posting per sub-range
        terms[t] = rng.choice(N, size=int(rng.integers(30, 150)), replace=False); t += 1
    for _ in range(4):            # sparse class overall, but 65-300 consecutive docs in a few sub-ranges
        subs = rng.choice(N_SUB, size=6, replace=False)
        docs = [s * S + int(rng.integers(0, S - 300)) + np.arange(int(rng.integers(65, 300))) for s in subs]
        terms[t] = np.concatenate(docs); t += 1
    for _ in range(5):            # dense-posting terms
        terms[t] = rng.choice(N, size=int(rng.integers(3500, 20000)), replace=False); t += 1
    terms[t] = rng.choice(N, size=int(0.25 * N), replace=False); t += 1     # a streamed row
    return terms


@pytest.fixture(scope="module")
def walk_corpus():
    rng = np.random.default_rng(20261020)
    terms = _designed_terms(rng)
    n_hot = len(terms)
    docs, toks = [], []
    for t, d in terms.items():
        reps = rng.integers(1, 4, size=d.size)              # tf 1..3
        docs.append(np.repeat(d, reps)); toks.append(np.full(int(reps.sum()), t, np.int32))
    fill = rng.integers(4, 12, size=N)
    docs.append(np.repeat(np.arange(N), fill))
    toks.append(rng.integers(n_hot, FILL_VOCAB, size=int(fill.sum())).astype(np.int32))
    d = np.concatenate(docs); tk = np.concatenate(toks)
    order = np.argsort(d, kind="stable")
    tok = tk[order]
    off = np.zeros(N + 1, np.int64)
    np.cumsum(np.bincount(d, minlength=N), out=off[1:])
    # queries: short ones (regular pass) mixing every class, with repeated terms, and long ones (21-32 hot terms:
    # the long-query pass)
    qs = []
    for i in range(240):
        n = int(rng.integers(2, 9))
        q = list(rng.choice(n_hot, size=n, replace=False))
        q += list(rng.choice(q, size=int(rng.integers(0, 3))))                         # duplicates
        q += list(rng.integers(n_hot, FILL_VOCAB, size=int(rng.integers(0, 3))))       # cold terms
        qs.append(q)
    for i in range(40):
        q = list(rng.choice(n_hot, size=int(rng.integers(21, n_hot)), replace=False))
        q += list(rng.choice(q, size=int(rng.integers(0, 3))))
        qs.append(q[:64])
    qo = np.zeros(len(qs) + 1, np.int32)
    np.cumsum([len(q) for q in qs], out=qo[1:])
    qt = np.asarray([t for q in qs for t in q], np.int32)
    return off, tok, qo, qt


@pytest.mark.parametrize("dedup", [True, False])
@pytest.mark.parametrize("defer_pm", [650, 0])
@pytest.mark.parametrize("k", [10, 100])
def test_walk_fused_equals_dense_and_oracle(walk_corpus, dedup, defer_pm, k):
    from document_retrieval_b200 import BM25
    off, tok, qo, qt = walk_corpus
    m = BM25.from_token_ids(off, tok, FILL_VOCAB, variant="okapi", dedup_query=dedup)
    m.set_option("defer_pm", defer_pm)          # 0: nothing deferred, the dense-posting terms are walked too
    q = (qt, qo)
    ids_f, sc_f = m.retrieve_top_n_batch(q, k)
    n_fused = m.query_stats()["queries_fused"]
    assert n_fused >= qo.size - 1 - 10
    m.set_option("fused_long", 0)
    m.retrieve_top_n_batch(q, k)
    assert m.query_stats()["queries_fused"] <= n_fused - 30          # the long queries did take the long pass
    m.set_option("fused_long", 1)
    m.set_option("fused", 0)
    ids_d, sc_d = m.retrieve_top_n_batch(q, k)
    m.set_option("fused", 1)
    assert torch.equal(ids_f, ids_d) and torch.equal(sc_f, sc_d)
    o = COracle(off, tok, FILL_VOCAB, variant="okapi")
    oi, osc, _ = o.topk_batch(qt, qo, k, dedup=dedup)
    assert np.array_equal(ids_f.cpu().numpy(), oi)
    assert np.array_equal(sc_f.cpu().numpy(), osc)
