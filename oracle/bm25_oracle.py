"""TEST INFRASTRUCTURE - CPU (numpy) restatement of the reference's BM25 / cosine hot path.

This module is the *checker*: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  The product
(``document_retrieval_b200``) never does and has no CPU fallback.

Parity pinning: the reference holds no golden vectors (SURVEY 4), so this restatement is pinned
against the *unmodified reference functions executed in the authoring container*
(``oracle/ref_loader.py``) - ``tests/golden/make_golden.py`` stores their outputs as the fixtures
under ``tests/golden/`` that ``tests/test_oracle.py`` checks this module against.

Every function cites the reference lines it restates.  Arithmetic is float64 with the
reference's own operation order, so per-posting contributions are bit-identical to the Python
scalars; the only freedom is the order in which a query's terms are summed (the reference
iterates ``set(query)``, i.e. hash order) - here it is ascending term id.

Variants (SURVEY appendix A):
  "notebook"        idf = ln(1 + (N-df+.5)/(df+.5)),  norm = 1 - b + dl/avgdl       (b NOT applied)
                    bm25_ranking.ipynb:189,202 ; final_implementation.py:116-118,142
  "okapi"           idf = ln((N-df+.5)/(df+.5) + 1),  norm = 1 - b + b*dl/avgdl
                    team_run1.py:187,193
  "okapi_no_plus1"  idf = ln((N-df+.5)/(df+.5)),      norm = 1 - b + b*dl/avgdl
                    cosine_similarity_bm25_reranking.py:179 (idf can be negative)
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

VARIANTS = ("notebook", "okapi", "okapi_no_plus1")


@dataclass
class OracleIndex:
    n_docs: int
    vocab: int
    row_ptr: np.ndarray   # int64[V+1]   CSR by term
    post_doc: np.ndarray  # int32[nnz]   doc ids ascending inside a term (bm25_ranking.ipynb:186)
    post_tf: np.ndarray   # int32[nnz]
    dl: np.ndarray        # int64[N]     token count per doc (= sum of tf, bm25_ranking.ipynb:201)
    df: np.ndarray        # int64[V]
    avgdl: float          # sum(len(doc))/N, bm25_ranking.ipynb:171


def build_index(doc_offsets: np.ndarray, token_ids: np.ndarray, vocab: int) -> OracleIndex:
    """BM25.build, bm25_ranking.ipynb:178-186 (tf per doc, df, postings in doc order).
    Tokens outside [0, vocab) are rejected - the corpus defines the vocabulary."""
    doc_offsets = np.asarray(doc_offsets, dtype=np.int64)
    token_ids = np.asarray(token_ids, dtype=np.int64)
    n_docs = doc_offsets.size - 1
    if token_ids.size and (token_ids.min() < 0 or token_ids.max() >= vocab):
        raise ValueError("token id outside [0, vocab)")
    dl = np.diff(doc_offsets)
    doc_of_tok = np.repeat(np.arange(n_docs, dtype=np.int64), dl)
    key = token_ids * n_docs + doc_of_tok               # (term, doc) -> sorted = CSR order
    uniq, tf = np.unique(key, return_counts=True)
    term = uniq // max(n_docs, 1)
    doc = uniq - term * n_docs
    df = np.bincount(term, minlength=vocab).astype(np.int64)
    row_ptr = np.zeros(vocab + 1, dtype=np.int64)
    np.cumsum(df, out=row_ptr[1:])
    total = int(dl.sum())
    avgdl = total / n_docs                               # ZeroDivisionError on empty corpus, like :171
    return OracleIndex(n_docs, vocab, row_ptr, doc.astype(np.int32), tf.astype(np.int32), dl, df, avgdl)


def idf_value(df: int, n_docs, variant: str) -> float:
    """bm25_ranking.ipynb:189 / team_run1.py:187 / cosine_similarity_bm25_reranking.py:179."""
    x = (n_docs - df + 0.5) / (df + 0.5)
    if variant == "notebook":
        return math.log(1 + x)
    if variant == "okapi":
        return math.log(x + 1)
    if variant == "okapi_no_plus1":
        return math.log(x)
    raise ValueError(variant)


def idf_table(df: np.ndarray, n_docs, variant: str) -> np.ndarray:
    """idf per term id; terms with df == 0 get NaN (they are not in the reference's dicts)."""
    out = np.full(df.size, np.nan, dtype=np.float64)
    for d in np.unique(df):
        if d > 0:
            out[df == d] = idf_value(int(d), n_docs, variant)
    return out


def _norm(dl, avgdl, b, variant):
    if variant == "notebook":
        return 1 - b + dl / avgdl                        # bm25_ranking.ipynb:202
    return 1 - b + b * dl / avgdl                        # team_run1.py:193


def term_contrib(ix: OracleIndex, t: int, idf_t: float, k1: float, b: float, variant: str,
                 n_docs=None, avgdl=None):
    """(docs, contribution[float64]) of one term - the body of the loop at
    bm25_ranking.ipynb:199-203:  idf * ((tf*(k1+1)) / (tf + k1*norm))."""
    lo, hi = int(ix.row_ptr[t]), int(ix.row_ptr[t + 1])
    docs = ix.post_doc[lo:hi]
    tf = ix.post_tf[lo:hi].astype(np.float64)
    dl = ix.dl[docs].astype(np.float64)
    avg = ix.avgdl if avgdl is None else avgdl
    return docs, idf_t * ((tf * (k1 + 1)) / (tf + k1 * _norm(dl, avg, b, variant)))


def get_scores(ix: OracleIndex, q_terms, variant="notebook", dedup=True, k1=1.5, b=0.75,
               n_docs=None, avgdl=None, df=None) -> np.ndarray:
    """BM25.get_scores, bm25_ranking.ipynb:191-204 (dedup=True: ``set(query)``), or the scoring
    loop of score_documents_for_query, team_run1.py:183-194 (dedup=False: duplicates counted, in
    query order).  OOV terms (outside the vocabulary or df == 0) are skipped (:195-196).
    ``n_docs``/``avgdl``/``df`` override the index's own statistics (global statistics of a
    doc-sharded corpus)."""
    N = ix.n_docs if n_docs is None else n_docs
    dfv = ix.df if df is None else df
    scores = np.zeros(ix.n_docs, dtype=np.float64)
    terms = [int(t) for t in q_terms if 0 <= int(t) < ix.vocab and dfv[int(t)] > 0]
    if dedup:
        terms = sorted(set(terms))
    for t in terms:
        docs, c = term_contrib(ix, t, idf_value(int(dfv[t]), N, variant), k1, b, variant, N, avgdl)
        scores[docs] += c                                # doc ids are unique inside one term
    return scores


def topk_canonical(scores: np.ndarray, k: int, positive_only: bool = False):
    """retrieve_top_n, bm25_ranking.ipynb:206-213, with the tie order made canonical: score
    descending, doc id ascending (the reference's argpartition/argsort order among equal
    scores is implementation-defined, SURVEY 8c).  ``positive_only`` restricts candidates to
    docs with >= 1 hit, like ``heapq.nlargest(100, scores)`` over the dict of touched docs
    (team_run1.py:196).  -> (ids int64[<=k], scores float64[<=k])"""
    n = scores.size
    ids = np.arange(n, dtype=np.int64)
    if positive_only:
        ids = ids[scores != 0.0]
    if k < ids.size:
        # exact cut: everything >= k-th largest value, then canonical order
        kth = np.partition(scores[ids], ids.size - k)[ids.size - k]
        ids = ids[scores[ids] >= kth]
    order = np.lexsort((ids, -scores[ids]))[:k]
    ids = ids[order]
    return ids, scores[ids]


def retrieve_top_n(ix: OracleIndex, q_terms, n=10, variant="notebook", dedup=True, k1=1.5, b=0.75,
                   **kw):
    return topk_canonical(get_scores(ix, q_terms, variant, dedup, k1, b, **kw), n)


def score_documents_for_query(ix: OracleIndex, q_terms, top=100, k1=1.5, b=0.75):
    """team_run1.py:173-199 - okapi variant, duplicates counted, only docs with a hit, top-100."""
    s = get_scores(ix, q_terms, "okapi", dedup=False, k1=k1, b=b)
    return topk_canonical(s, top, positive_only=True)


def bm25_score_rerank(ix: OracleIndex, q_terms, doc: int, idf: np.ndarray, avgdl: float,
                      k1=1.5, b=0.75) -> float:
    """bm25_score, cosine_similarity_bm25_reranking.py:185-195 - the "V3" re-rank formula:
    ``doc_length`` is the sum of the query terms' tf in this doc (:187), duplicates counted, idf
    taken from ``idf`` (no +1 in compute_idf :179).  Terms absent from the corpus are skipped
    (``if term in tf_dict``)."""
    def tf_of(t):
        if not (0 <= t < ix.vocab):
            return None
        lo, hi = int(ix.row_ptr[t]), int(ix.row_ptr[t + 1])
        if lo == hi:
            return None
        j = lo + int(np.searchsorted(ix.post_doc[lo:hi], doc))
        return int(ix.post_tf[j]) if j < hi and ix.post_doc[j] == doc else 0
    tfs = [tf_of(int(t)) for t in q_terms]
    doc_length = sum(tf for tf in tfs if tf)
    score = 0
    for t, tf in zip(q_terms, tfs):
        if tf is None:
            continue
        numerator = tf * (k1 + 1)
        denominator = tf + k1 * (1 - b + b * (doc_length / avgdl))
        score += float(idf[int(t)]) * (numerator / denominator)
    return score


def recall_at_k(retrieved, positives) -> float:
    """evaluate_recall_at_k, bm25_ranking.ipynb:329-354: hits / len(val); a skipped query
    (``retrieved[i] is None``) still counts in the denominator (:331,353)."""
    total = len(positives)
    hits = sum(1 for r, p in zip(retrieved, positives) if r is not None and p in list(r))
    return hits / total if total > 0 else 0


def mrr_recall_at_k(ranked, relevant, k):
    """team_run1.py:307-318 for one query."""
    top = list(ranked)[:k]
    mrr = 0.0
    for i, d in enumerate(top):
        if d in relevant:
            mrr = 1 / (i + 1)
            break
    rec = len(set(relevant) & set(top)) / len(relevant)
    return mrr, rec


def cosine_topk(doc_emb, query_emb, k: int):
    """Dense cosine re-rank, team_run1.py:270-282: e/(||e||+1e-10) on both sides (fp32), matmul,
    topk.  Ties canonicalised by doc id.  Inputs are float32 [N,D] / [Q,D] arrays (bf16 data is
    widened by the caller).  -> (ids int64[Q,k], sims float32[Q,k])"""
    import torch
    d = torch.as_tensor(np.asarray(doc_emb, dtype=np.float32))
    q = torch.as_tensor(np.asarray(query_emb, dtype=np.float32))
    d = d / (d.norm(dim=1, keepdim=True) + 1e-10)
    q = q / (q.norm(dim=1, keepdim=True) + 1e-10)
    sims = torch.matmul(q, d.T).numpy()
    ids = np.empty((sims.shape[0], k), dtype=np.int64)
    val = np.empty((sims.shape[0], k), dtype=np.float32)
    for i in range(sims.shape[0]):
        o = np.lexsort((np.arange(sims.shape[1]), -sims[i]))[:k]
        ids[i], val[i] = o, sims[i, o]
    return ids, val


def tfidf_cosine_scores(ix: OracleIndex, q_terms, idf: np.ndarray) -> np.ndarray:
    """Sparse TF-IDF cosine of one query against every doc, cosine_similarity_bm25_reranking.py:72-110,121-126,
    210-226, with the reference's mixed precision (probed with scipy 1.18): doc vector ``float32(tf * idf)``
    (lil_matrix float32, :88); ``doc_norms`` float64 (sqrt of the float64 sum of squares, :210); query vector
    ``float32(idf)`` per DISTINCT in-corpus term (set, not add, :121-126) times the float32 scalar ``1/norm(q)``
    (:222-223); the product ``normalized.dot(q.T)`` is float64 (:226).  A zero-norm doc gives 0.  -> float64[N]"""
    ts = np.unique(np.asarray([int(t) for t in q_terms if 0 <= int(t) < ix.vocab and ix.row_ptr[int(t) + 1] > ix.row_ptr[int(t)]],
                              dtype=np.int64))
    out = np.zeros(ix.n_docs, np.float64)
    if ts.size == 0:
        return out
    q = idf[ts].astype(np.float32)
    qnorm = np.linalg.norm(q)           # float32, what scipy.sparse.linalg.norm returns for the float32 query row (BLAS sdot)
    qn = (q * np.float32(np.float32(1.0) / qnorm)).astype(np.float32)
    norm2 = doc_sq_norms(ix, idf)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = 1.0 / np.sqrt(norm2)
    for j, t in enumerate(ts):                                   # ascending term id
        lo, hi = int(ix.row_ptr[t]), int(ix.row_ptr[t + 1])
        d = ix.post_doc[lo:hi]
        e = (ix.post_tf[lo:hi].astype(np.float64) * float(idf[t])).astype(np.float32).astype(np.float64)
        out[d] += (e * inv[d]) * float(qn[j])
    return np.nan_to_num(out, nan=0.0, posinf=0.0, neginf=0.0)


def doc_sq_norms(ix: OracleIndex, idf: np.ndarray) -> np.ndarray:
    """float64 sum over the doc's terms of float32(tf*idf)^2 (the square of ``doc_norms``, :210)."""
    cache = getattr(ix, "_sq_norms", None)
    if cache is not None and cache[0] is idf:
        return cache[1]
    term_of = np.repeat(np.arange(ix.vocab), np.diff(ix.row_ptr))
    e = (ix.post_tf.astype(np.float64) * np.nan_to_num(idf[term_of])).astype(np.float32).astype(np.float64)
    n2 = np.zeros(ix.n_docs, np.float64)
    np.add.at(n2, ix.post_doc, e * e)
    try:
        ix._sq_norms = (idf, n2)
    except Exception:
        pass
    return n2


def rank_cosine_then_bm25(ix: OracleIndex, queries, idf: np.ndarray, avgdl: float, n_candidates=200, k=10,
                          doc_lang=None, query_lang=None):
    """rank_documents_with_cosine_similarity_and_bm25, cosine_similarity_bm25_reranking.py:198-238: cosine over the
    whole corpus -> first ``n_candidates`` of the descending order (:229; canonical order (cosine desc, doc id asc)) ->
    bm25_score of the candidates (:232-233) -> stable descending sort, first ``k`` (:234).  With ``doc_lang`` /
    ``query_lang`` the candidates are the first ``n_candidates`` docs OF THE QUERY'S LANGUAGE in that order
    (text_preprocessing_and_embedding_setup.py:333-343; there n_candidates = 1000 and k = 100, :349).
    ``queries`` is a list of term-id lists.  -> list of (ids int64[<=k], cand ids, cand cosines)"""
    out = []
    ids = np.arange(ix.n_docs)
    for i, q in enumerate(queries):
        cos = tfidf_cosine_scores(ix, q, idf)
        order = np.lexsort((ids, -cos))
        if doc_lang is not None:
            order = order[np.asarray(doc_lang)[order] == query_lang[i]]
        cand = order[:n_candidates]
        sc = np.array([bm25_score_rerank(ix, q, int(d), idf, avgdl) for d in cand], dtype=np.float64)
        o = np.argsort(-sc, kind="stable")[:k]
        out.append((cand[o].astype(np.int64), cand.astype(np.int64), cos[cand]))
    return out


def per_language_recall(ranked_docs, positives, query_langs):
    """text_preprocessing_and_embedding_setup.py:534-562: overall hit rate and hits / queries per language."""
    per_q, per_hit = {}, {}
    hits = 0
    for r, p, lang in zip(ranked_docs, positives, query_langs):
        per_q[lang] = per_q.get(lang, 0) + 1
        per_hit.setdefault(lang, 0)
        if p in list(r):
            hits += 1
            per_hit[lang] += 1
    n = len(positives)
    return (hits / n if n else 0), {lang: per_hit[lang] / per_q[lang] for lang in per_q}
