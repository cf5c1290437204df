"""BM25 top-k under okapi_no_plus1 (idf = ln((N-df+.5)/(df+.5)), negative for df > N/2) against the float64 oracle, bit
for bit, where the fp32 sums of the dense path cancel.

A query with a term of negative idf sums weights of both signs.  A doc's fp32 sum can then be exactly 0 while its float64
score is not (and a float64 score can be ~1e-7 from 0 while fp32 rounds it away), so neither "fp32 score 0 means no hit"
nor a band relative to the k-th fp32 score is safe.  The designed corpora below plant docs whose two query-term weights
cancel to an fp32 sum of exactly 0 with a float64 score of a chosen sign: the sum of doc lengths (through avgdl) is solved
on the host so that w_A + w_B crosses 0 at the designed doc.  Every test first checks on the device that the design still
holds (br_score_batch returns exactly 0.0 there), so it fails rather than passing once it stops covering the edge."""
import math

import numpy as np
import pytest
import torch

from oracle import bm25_oracle as orc

K1, B = 1.5, 0.75
VARIANT = "okapi_no_plus1"


# ------------------------------------------------------------------------------------------------ design helper (CPU)
def idf(df, n):
    return math.log((n - df + 0.5) / (df + 0.5))


def weight(idf_t, tf, dl, sum_dl, n):
    """float64 posting weight in the operation order of the oracle and of the library (bm25_contrib)."""
    norm = (1.0 - B) + (B * dl) / (sum_dl / n)
    return idf_t * ((tf * (K1 + 1.0)) / (tf + K1 * norm))


def emulate(n, df_a, df_b, tf_a, tf_b, dl, sum_dl):
    """(float64 score, fp32 score) of a doc holding both terms: each weight rounded to fp32 as k_weights does, then one
    fp32 add (two terms: the order of the atomic adds does not matter)."""
    wa = weight(idf(df_a, n), tf_a, dl, sum_dl, n)
    wb = weight(idf(df_b, n), tf_b, dl, sum_dl, n)
    return wb + wa, float(np.float32(np.float32(wb) + np.float32(wa)))


def find_designs(n, df_a, df_b, sign, sum_dl_range=None, tf_a_max=60, tf_b_max=4, n_dl=80):
    """Designs (tf_a, tf_b, dl, sum_dl, s64) with an fp32 sum of exactly 0 and a float64 score of the given sign.  For
    every (tf_a, tf_b, dl) the sum of doc lengths that puts w_A + w_B at 0 is found by bisection; the integers around it
    are checked."""
    lo_s, hi_s = sum_dl_range or (0, 1000 * n)
    out = []
    for tf_a in range(2, tf_a_max):
        for tf_b in range(1, tf_b_max + 1):
            for dl in range(tf_a + tf_b, tf_a + tf_b + n_dl):
                f = lambda s: emulate(n, df_a, df_b, tf_a, tf_b, dl, s)[0]
                a, c = max(lo_s, dl + n - 1), hi_s
                if a >= c or f(a) * f(c) > 0:
                    continue
                while c - a > 1:
                    m = (a + c) // 2
                    if (f(m) > 0) == (f(a) > 0):
                        a = m
                    else:
                        c = m
                for s in range(a - 2, a + 3):
                    s64, s32 = emulate(n, df_a, df_b, tf_a, tf_b, dl, s)
                    if s32 == 0.0 and np.sign(s64) == sign and lo_s <= s <= hi_s:
                        out.append((tf_a, tf_b, dl, s, s64))
    return out


def test_design_helper_reproduces_the_cancellations():
    """N = 1000, df_A = 900 (idf -2.19), df_B = 2: the two documented rows, and the counts of the scan."""
    s64, s32 = emulate(1000, 900, 2, 9, 1, 33, 17584)
    assert s32 == 0.0 and s64 == 2.4497676331947105e-07
    s64, s32 = emulate(1000, 900, 2, 5, 1, 70, 22879)
    assert s32 == 0.0 and s64 == -1.8566204618153392e-07
    pos, neg = find_designs(1000, 900, 2, +1), find_designs(1000, 900, 2, -1)
    assert (9, 1, 33, 17584, 2.4497676331947105e-07) in pos and (5, 1, 70, 22879, -1.8566204618153392e-07) in neg
    assert (len(pos), len(neg)) == (47, 42)
    assert idf(900, 1000) < 0 < idf(2, 1000) and idf(500, 1000) == 0.0


# ------------------------------------------------------------------------------------------------ corpus builder
def positions(start, counts):
    """Token positions start[d] .. start[d] + counts[d] - 1 of every doc d, concatenated."""
    counts = np.asarray(counts, np.int64)
    first = np.repeat(np.cumsum(counts) - counts, counts)
    return np.repeat(np.asarray(start, np.int64), counts) + np.arange(int(counts.sum())) - first


def build_corpus(n, tf, fixed_dl, sum_dl, n_fill, seed):
    """Docs of the given per-term tf ({term: int64[N]}), with filler tokens (terms >= 16, small df) making up the
    lengths: docs in fixed_dl ({doc: dl}) get exactly that length, the others at least one filler token, and the
    remainder of sum_dl is spread over them at random.  -> (doc_offsets, token_ids)"""
    rng = np.random.Generator(np.random.PCG64(seed))
    need = sum(tf.values())
    dl = need.copy()
    free = np.ones(n, bool)
    for d, L in fixed_dl.items():
        assert L >= need[d]
        dl[d] = L
        free[d] = False
    dl[free] += 1
    rest = sum_dl - int(dl.sum())
    assert rest >= 0, (sum_dl, int(dl.sum()))
    dl[np.nonzero(free)[0]] += np.bincount(rng.integers(0, int(free.sum()), rest), minlength=int(free.sum()))
    off = np.zeros(n + 1, np.int64)
    np.cumsum(dl, out=off[1:])
    assert off[-1] == sum_dl
    tok = rng.integers(16, 16 + n_fill, int(sum_dl)).astype(np.int32)
    start = off[:-1].copy()
    for t, c in tf.items():
        tok[positions(start, c)] = t
        start += c
    return off, tok


def pick_design(n, df_a, df_b, sign, base_len, max_avgdl):
    """The first design whose sum of doc lengths leaves room for the other docs (base_len tokens at least)."""
    for d in find_designs(n, df_a, df_b, sign, (base_len + 200, int(max_avgdl * n))):
        if d[3] - 2 * d[2] >= base_len:
            return d
    raise AssertionError("no design found")


# ------------------------------------------------------------------------------------------------ 1a. designed corpora
A, BT, Z, OOV = 0, 1, 2, 10_000
N_A = 1000
DESIGNED = (0, 40)                    # doc 0: below every no-hit doc; doc 40: above the no-hit docs 1..39
B_ONLY = 41                           # the one positive doc of [A, B] besides the designed ones
A_ONLY = np.arange(42, 940)           # negative scores; 940..999 are no-hit docs again
QUERIES = [[A, BT], [BT, A], [A, BT, OOV, -1], [A], [BT], [A, BT, BT], [Z], [Z, A], [Z, BT], [A, BT, Z]]
CANCEL = (0, 1, 2, 9)                 # queries whose fp32 sum cancels at the designed docs (with dedup, also query 5)


def designed_corpus(sign):
    """N = 1000: term A (df 900, idf < 0), term B (df 3, idf > 0) in the two designed docs and in B_ONLY, term Z on the
    even doc ids (df = N/2, idf exactly 0)."""
    n = N_A
    rng = np.random.Generator(np.random.PCG64(7 + sign))
    tf_a = np.zeros(n, np.int64)
    tf_a[A_ONLY] = rng.integers(1, 4, A_ONLY.size)
    tf_b = np.zeros(n, np.int64)
    tf_b[B_ONLY] = 1
    tf_z = np.zeros(n, np.int64)
    tf_z[::2] = 1
    base = int((tf_a + tf_b + tf_z).sum()) + n
    d = pick_design(n, 900, 3, sign, base, 30)
    for doc in DESIGNED:
        tf_a[doc], tf_b[doc] = d[0], d[1]
    assert (tf_a > 0).sum() == 900 and (tf_b > 0).sum() == 3 and (tf_z > 0).sum() == n // 2
    off, tok = build_corpus(n, {A: tf_a, BT: tf_b, Z: tf_z}, {doc: d[2] for doc in DESIGNED}, d[3], 2000, 11 + sign)
    return off, tok, d


def pack(queries):
    q_off = np.zeros(len(queries) + 1, np.int32)
    np.cumsum([len(q) for q in queries], out=q_off[1:])
    return np.asarray([t for q in queries for t in q], np.int32), q_off


def canonical(scores, k, positive_only, allowed=None):
    """Oracle top-k of the allowed docs, padded to k: (ids, scores, count)."""
    docs = np.arange(scores.size) if allowed is None else np.nonzero(allowed)[0]
    li, ls = orc.topk_canonical(scores[docs], k, positive_only)
    ids = np.full(k, -1, np.int64)
    sc = np.zeros(k, np.float64)
    ids[:li.size], sc[:li.size] = docs[li], ls
    return ids, sc, li.size


def check_design(m, co, queries, cancel, designed, sign, dedup):
    """br_score_batch (k_score_dense, the dense path's scorer) gives exactly 0.0 at the designed docs, and the oracle's
    float64 score there has the designed sign."""
    s32 = m.get_scores_batch(pack(queries)).cpu().numpy()
    for i in cancel:
        s64 = co.get_scores(queries[i], dedup)
        for doc in designed:
            assert s32[i, doc] == 0.0, ("design lost: fp32 score is not 0", i, doc, s32[i, doc])
            assert np.sign(s64[doc]) == sign, ("design lost: float64 sign", i, doc, s64[doc])


def special_ks(oracle_scores, n):
    ks = {1, 2, 1024}
    for s in oracle_scores:
        n_pos, n_nonneg = int((s > 0).sum()), int((s >= 0).sum())
        ks |= {n_pos, n_pos + 1, n_nonneg - 1, n_nonneg, n_nonneg + 1}
    return sorted(k for k in ks if 1 <= k <= 1024)


def fake_shards(off, tok, vocab, bounds, dedup):
    from document_retrieval_b200 import BM25
    shards = []
    for lo, hi in bounds:
        shards.append(BM25.from_token_ids(off[lo:hi + 1] - off[lo], tok[off[lo]:off[hi]], vocab, variant=VARIANT,
                                          dedup_query=dedup, doc_base=lo, finalize=False))
    df = sum(s.local_df_tensor().to(torch.int64) for s in shards).cpu().numpy()
    for s in shards:
        s.finalize(off.size - 1, int(off[-1]), df)
    return shards


@pytest.fixture(scope="module", params=[+1, -1], ids=["fp32_zero_float64_pos", "fp32_zero_float64_neg"])
def designed(request):
    from oracle.c_oracle import COracle
    off, tok, d = designed_corpus(request.param)
    vocab = int(tok.max()) + 1
    return request.param, off, tok, vocab, d, COracle(off, tok, vocab, K1, B, VARIANT)


@pytest.mark.gpu
@pytest.mark.parametrize("dedup", [True, False])
def test_designed_cancellation_top_k(designed, dedup):
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.sharded import merge_topk_cuda
    sign, off, tok, vocab, d, co = designed
    n = off.size - 1
    m = BM25.from_token_ids(off, tok, vocab, variant=VARIANT, dedup_query=dedup)
    check_design(m, co, QUERIES, CANCEL + (() if not dedup else (5,)), DESIGNED, sign, dedup)
    q = pack(QUERIES)
    s64 = [co.get_scores(x, dedup) for x in QUERIES]
    nohit = np.setdiff1d(np.arange(n), np.concatenate([DESIGNED, [B_ONLY], A_ONLY]))       # no hit for [A, B]
    rows = np.ones((3, n), bool)
    rows[1, nohit[:5]] = False                                  # the lowest-id no-hit docs excluded
    rows[2] = False
    rows[2, [*DESIGNED, B_ONLY, nohit[0], nohit[-1], A_ONLY[0], A_ONLY[-1]]] = True      # 7 docs: fewer than most k
    shard_sets = {w: fake_shards(off, tok, vocab, b, dedup)
                  for w, b in ((2, [(0, 1), (1, n)]), (3, [(0, 1), (1, 40), (40, n)]))}
    for positive_only in (False, True):
        for k in special_ks(s64, n):
            want = [canonical(s, k, positive_only) for s in s64]
            ids, sc, cnt = (x.cpu().numpy() for x in m.retrieve_top_n_batch(q, k, positive_only, return_counts=True))
            for i, (oi, os_, oc) in enumerate(want):
                assert np.array_equal(ids[i], oi), (sign, dedup, positive_only, k, QUERIES[i], ids[i][:8], oi[:8])
                assert np.array_equal(sc[i], os_), (sign, dedup, positive_only, k, QUERIES[i])
                assert cnt[i] == oc, (sign, dedup, positive_only, k, QUERIES[i], cnt[i], oc)
            rec = m.retrieve_records_batch(q, k, positive_only).cpu()
            assert np.array_equal(rec[..., 0].numpy(), ids.astype(np.int64))
            assert np.array_equal(rec[..., 1].contiguous().view(torch.float64).numpy(), sc)
            for r in range(3):
                qrow = np.full(len(QUERIES), r, np.int32)
                fi, fs, fc = (x.cpu().numpy() for x in m.retrieve_top_n_batch(
                    q, k, positive_only, return_counts=True, doc_filter=rows, query_filter=qrow))
                if r == 0:                                      # all-ones row: the unfiltered call, bit for bit
                    assert np.array_equal(fi, ids) and np.array_equal(fs, sc) and np.array_equal(fc, cnt)
                for i, s in enumerate(s64):
                    oi, os_, oc = canonical(s, k, positive_only, rows[r])
                    assert np.array_equal(fi[i], oi) and np.array_equal(fs[i], os_) and fc[i] == oc, \
                        (sign, dedup, positive_only, k, r, QUERIES[i], fi[i][:8], oi[:8])
            for world, shards in shard_sets.items():
                parts_i, parts_s = [], []
                for s in shards:
                    si, ss = s.retrieve_top_n_batch(q, k, positive_only)
                    parts_i.append(torch.where(si >= 0, si.to(torch.int64) + s.doc_base, torch.full_like(si, -1, dtype=torch.int64)))
                    parts_s.append(ss)
                mi, ms = merge_topk_cuda(torch.stack(parts_i), torch.stack(parts_s), k)
                assert np.array_equal(mi.cpu().numpy(), ids.astype(np.int64)), (world, sign, dedup, positive_only, k)
                assert np.array_equal(ms.cpu().numpy(), sc), (world, sign, dedup, positive_only, k)
    for i, x in enumerate(QUERIES):                             # n >= N: the full ranking
        full, _, c = canonical(s64[i], n, False)
        assert np.array_equal(m.retrieve_top_n(np.asarray(x, np.int32), n + 3), full[:c]), (sign, dedup, x)


@pytest.mark.gpu
def test_designed_cancellation_fp32_scores_within_the_mixed_sign_bound(designed):
    """br_score_batch: |s32 - s64| <= (n + 2) 2^-24 sum_t mult_t |w_t,d| per doc, n the query's distinct terms."""
    from document_retrieval_b200 import BM25
    sign, off, tok, vocab, d, co = designed
    m = BM25.from_token_ids(off, tok, vocab, variant=VARIANT, dedup_query=False)
    check_mixed_sign_bound(m, co, off, tok, vocab, QUERIES, dedup=False)


def check_mixed_sign_bound(m, co, off, tok, vocab, queries, dedup):
    ix = orc.build_index(off, tok, vocab)
    s32 = m.get_scores_batch(pack(queries)).cpu().numpy().astype(np.float64)
    for i, x in enumerate(queries):
        terms = [t for t in x if 0 <= t < vocab and ix.df[t] > 0]
        mult = {t: (1 if dedup else terms.count(t)) for t in set(terms)}
        absw = np.zeros(ix.n_docs)
        for t, mt in mult.items():
            docs, c = orc.term_contrib(ix, t, orc.idf_value(int(ix.df[t]), ix.n_docs, VARIANT), K1, B, VARIANT)
            absw[docs] += mt * np.abs(c)
        s64 = co.get_scores(x, dedup)
        bound = (len(mult) + 2) * 2.0 ** -24 * absw
        err = np.abs(s32[i] - s64)
        assert (err <= bound).all(), (x, int(np.argmax(err - bound)), float((err - bound).max()))


# ------------------------------------------------------------------------------------------------ 1b. several dense passes
N_BIG = 2_000_000


@pytest.mark.gpu
def test_designed_cancellation_across_dense_passes():
    """2M docs: the dense path serves 2^30 / (4N) = 134 queries per pass, so 330 queries take three passes; the
    cancelling queries sit at the first and last slot of every pass (the q_begin offsets of select, emit and re-score)."""
    from document_retrieval_b200 import BM25
    from oracle.c_oracle import COracle
    n = N_BIG
    rng = np.random.Generator(np.random.PCG64(21))
    designed_docs = (3, 1_200_000)
    b_only = 1_500_000
    tf_a = np.zeros(n, np.int64)
    a_docs = rng.permutation(np.setdiff1d(np.arange(n), [*designed_docs, b_only]))[:1_800_000 - 2]
    tf_a[a_docs] = rng.integers(1, 3, a_docs.size)
    tf_b = np.zeros(n, np.int64)
    tf_b[b_only] = 1
    base = int((tf_a + tf_b).sum()) + n
    d = pick_design(n, 1_800_000, 3, +1, base, 8)
    for doc in designed_docs:
        tf_a[doc], tf_b[doc] = d[0], d[1]
    assert (tf_a > 0).sum() == 1_800_000 and (tf_b > 0).sum() == 3
    off, tok = build_corpus(n, {A: tf_a, BT: tf_b}, {doc: d[2] for doc in designed_docs}, d[3], 200_000, 22)
    vocab = int(tok.max()) + 1
    co = COracle(off, tok, vocab, K1, B, VARIANT)
    m = BM25.from_token_ids(off, tok, vocab, variant=VARIANT, dedup_query=True)
    distinct = [[A, BT], [BT, A, vocab + 5], [A], [A, 17, 18], [BT, 19], [A, BT, 20]]
    check_design(m, co, distinct, (0, 1), designed_docs, +1, True)
    qb = (1 << 30) // (4 * n)
    nq = 2 * qb + 62
    which = np.asarray([i % len(distinct) for i in range(nq)])
    for p in range(3):                                          # first and last query of every pass cancel
        which[p * qb] = 0
        which[min((p + 1) * qb, nq) - 1] = 1
    queries = [distinct[j] for j in which]
    s64 = [co.get_scores(x, True) for x in distinct]
    assert int(((tf_a == 0) & (tf_b == 0)).sum()) > 100_000                # a long zero-score tail of no-hit docs
    for positive_only in (False, True):
        for k in (1, 3, 4, 1000):
            ids, sc, cnt = (x.cpu().numpy() for x in m.retrieve_top_n_batch(pack(queries), k, positive_only, return_counts=True))
            for j, x in enumerate(distinct):
                oi, os_, oc = canonical(s64[j], k, positive_only)
                for i in np.nonzero(which == j)[0]:
                    assert np.array_equal(ids[i], oi), (positive_only, k, i, x, ids[i][:6], oi[:6])
                    assert np.array_equal(sc[i], os_) and cnt[i] == oc, (positive_only, k, i, x)
    assert m.query_stats()["queries_dense"] == nq


# ------------------------------------------------------------------------------------------------ 1c. random mixed signs
@pytest.fixture(scope="module")
def c1_mixed():
    from document_retrieval_b200 import synth
    from oracle.c_oracle import COracle
    c = synth.make_config("C1")
    n = c["n_docs"]
    df = np.diff(orc.build_index(c["doc_offsets"], c["token_ids"], c["vocab"]).row_ptr)
    neg = np.nonzero(df > n // 2 + (n % 2))[0]          # idf < 0
    pos = np.nonzero((df > 0) & (df < n // 2))[0]
    assert neg.size >= 3 and pos.size > 1000
    rng = np.random.Generator(np.random.PCG64(31))
    queries = []
    for i in range(240):
        L = int(rng.integers(3, 9))
        q = [int(rng.choice(neg)), int(rng.choice(pos[:300] if i % 2 else pos))]
        q += [int(rng.choice(neg if rng.random() < 0.4 else pos)) for _ in range(L - 2)]
        if i % 3 == 0:
            q.append(q[int(rng.integers(0, len(q)))])              # a duplicate
        queries.append([int(t) for t in rng.permutation(q)])
    return c, queries, COracle(c["doc_offsets"], c["token_ids"], c["vocab"], K1, B, VARIANT)


@pytest.mark.gpu
@pytest.mark.parametrize("dedup", [True, False])
def test_random_mixed_sign_queries_on_c1(c1_mixed, dedup):
    from document_retrieval_b200 import BM25
    c, queries, co = c1_mixed
    m = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], variant=VARIANT, dedup_query=dedup)
    q = pack(queries)
    s64 = [co.get_scores(x, dedup) for x in queries]
    for positive_only in (False, True):
        for k in (10, 100, 1000):
            ids, sc, cnt = (x.cpu().numpy() for x in m.retrieve_top_n_batch(q, k, positive_only, return_counts=True))
            for i, s in enumerate(s64):
                oi, os_, oc = canonical(s, k, positive_only)
                assert np.array_equal(ids[i], oi), (dedup, positive_only, k, queries[i])
                assert np.array_equal(sc[i], os_) and cnt[i] == oc, (dedup, positive_only, k, queries[i])
    assert m.query_stats()["queries_fused"] == 0                 # okapi_no_plus1 is served by the dense path only
    check_mixed_sign_bound(m, co, c["doc_offsets"], c["token_ids"], c["vocab"], queries[:40], dedup)


# ------------------------------------------------------------------------------------------------ idf exactly 0
@pytest.mark.gpu
def test_positive_only_drops_docs_whose_float64_score_is_zero():
    """df = N/2 gives idf = ln(1) = 0: a doc whose only hit is that term has a matching posting but scores exactly 0.
    positive_only keeps the docs whose float64 score is not 0, so it drops such docs, with or without a negative term in
    the query; positive_only = 0 ranks them with the no-hit docs, by doc id."""
    from document_retrieval_b200 import BM25
    n = 64
    docs = [[2] if d % 2 else [3, 3] for d in range(n)]          # term 2: df 32 = N/2
    for d in range(0, n, 3):
        docs[d].append(0)                                       # term 0: df 22, idf > 0
    for d in range(1, n, 5):
        docs[d] += [1] * (1 + d % 3)                            # term 1: df 13
    for d in range(40):
        docs[d].append(4)                                       # term 4: df 40 > N/2, idf < 0
    off = np.zeros(n + 1, np.int64)
    np.cumsum([len(x) for x in docs], out=off[1:])
    tok = np.asarray([t for x in docs for t in x], np.int32)
    ix = orc.build_index(off, tok, 5)
    assert ix.df[2] == n // 2 and orc.idf_value(int(ix.df[2]), n, VARIANT) == 0.0
    m = BM25.from_token_ids(off, tok, 5, variant=VARIANT)
    queries = [[2], [2, 0], [2, 4], [2, 0, 4], [2, 1, 4]]
    for k in (1, 5, 20, 40, 64):
        for positive_only in (False, True):
            ids, sc, cnt = (x.cpu().numpy() for x in m.retrieve_top_n_batch(pack(queries), k, positive_only, return_counts=True))
            for i, x in enumerate(queries):
                oi, os_, oc = canonical(orc.get_scores(ix, x, VARIANT), k, positive_only)
                assert np.array_equal(ids[i], oi) and np.array_equal(sc[i], os_) and cnt[i] == oc, (k, positive_only, x)
    ids, _, cnt = m.retrieve_top_n_batch(pack([[2]]), 10, True, return_counts=True)
    assert int(cnt[0]) == 0 and (ids == -1).all()
