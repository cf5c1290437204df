"""Hybrid retrieval: BM25 and dense cosine candidates fused into one ranking, by reciprocal rank (RRF) or by a convex
combination of per-query min-max-normalised exact scores.  Both fusions run in libbr_b200.so (br_fuse_rrf,
br_fuse_linear); host code here only moves tensors.

Candidate lists are [Q, n] int tensors of the BM25 index's LOCAL doc ids, -1 = empty slot.  A doc's rank in a list is
1 + the slot of its first occurrence.  Results are ordered by (fused score desc, doc id asc), -1 / 0.0 pad when the union
of the two lists has fewer than k members."""
from __future__ import annotations

import torch

from . import _lib
from ._lib import check, ptr
from .cosine import _bf16

MAX_DENSE = 256   # k limit of the cosine top-k


def _ids(x, dev, what):
    t = torch.as_tensor(x)
    if t.dim() != 2:
        raise ValueError(f"{what} must be [Q, n], got shape {tuple(t.shape)}")
    if t.dtype.is_floating_point or t.dtype == torch.bool:
        raise ValueError(f"{what} must be an integer array, got {t.dtype}")
    t = t.to(dev)
    if t.dtype != torch.int32 and t.numel() and (int(t.min()) < -2 ** 31 or int(t.max()) >= 2 ** 31):
        raise ValueError(f"{what} values must fit int32")
    return t.to(torch.int32).contiguous()


def _lists(bm25_ids, dense_ids, dev):
    b, d = _ids(bm25_ids, dev, "bm25_ids"), _ids(dense_ids, dev, "dense_ids")
    if b.shape[0] != d.shape[0]:
        raise ValueError(f"bm25_ids has {b.shape[0]} queries, dense_ids {d.shape[0]}")
    return b, d


def _check_k(k):
    k = int(k)
    if not 1 <= k <= _lib.BR_MAX_K:
        raise ValueError(f"k must be in [1, {_lib.BR_MAX_K}]")
    return k


def _check_docs(bm25_model, cosine_index):
    """The cosine side must cover the BM25 documents: one row per doc (flat) or one group per doc (grouped)."""
    if cosine_index.row_group is None:
        if cosine_index.n_docs != bm25_model.corpus_size:
            raise ValueError(f"the cosine index has {cosine_index.n_docs} rows, the BM25 model {bm25_model.corpus_size} "
                             "documents: without row_group the rows must be the BM25 documents")
    elif cosine_index.n_groups != bm25_model.corpus_size:
        raise ValueError(f"the cosine index has {cosine_index.n_groups} groups, the BM25 model {bm25_model.corpus_size} "
                         "documents: the groups must be the BM25 documents")


def fuse_rrf(bm25_ids, dense_ids, n_docs, k=10, rrf_c=60.0, weights=(1.0, 1.0)):
    """Reciprocal rank fusion of two candidate lists over ids in [0, n_docs): f(d) = w_bm25 / (rrf_c + r_b(d)) +
    w_dense / (rrf_c + r_d(d)), a term omitted when d is absent from that list, float64 -> (ids int32[Q, k], scores
    float64[Q, k]) on the device.  An id outside [-1, n_docs), a negative or non-finite rrf_c or weight, or both weights 0
    raise BRError."""
    lib = _lib.load()
    k = _check_k(k)
    w_b, w_d = (float(w) for w in weights)
    dev = bm25_ids.device if torch.is_tensor(bm25_ids) and bm25_ids.is_cuda else _lib.require_cuda()
    with torch.cuda.device(dev):
        b, d = _lists(bm25_ids, dense_ids, dev)
        nq = b.shape[0]
        ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
        sc = torch.empty((nq, k), dtype=torch.float64, device=dev)
        check(lib.br_fuse_rrf(ptr(b), b.shape[1], ptr(d), d.shape[1], int(n_docs), nq, float(rrf_c), w_b, w_d, k, ptr(ids),
                              ptr(sc), None, _lib.stream_ptr(dev)), "br_fuse_rrf")
    return ids, sc


def _fuse_linear_packed(bm25_model, cosine_index, q_terms, q_off, query_embeddings, bm25_ids, dense_ids, k, alpha):
    bm25_model._require()
    lib = _lib.load()
    k = _check_k(k)
    _check_docs(bm25_model, cosine_index)
    dev = bm25_model._device
    nq = q_off.numel() - 1
    qe = _bf16(query_embeddings, dev)
    if qe.dim() != 2 or qe.shape[0] != nq:
        raise ValueError(f"query_embeddings must be [{nq}, d] (one row per query), got {tuple(qe.shape)}")
    with torch.cuda.device(dev):
        b, d = _lists(bm25_ids, dense_ids, dev)
        if b.shape[0] != nq:
            raise ValueError(f"the candidate lists have {b.shape[0]} queries, the batch {nq}")
        ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
        sc = torch.empty((nq, k), dtype=torch.float64, device=dev)
        s_b = torch.empty((nq, k), dtype=torch.float64, device=dev)
        s_c = torch.empty((nq, k), dtype=torch.float32, device=dev)
        ci = cosine_index
        check(lib.br_fuse_linear(bm25_model._h, ptr(q_terms), ptr(q_off), nq, int(q_terms.numel()),
                                 int(bm25_model.dedup_query), ptr(ci.docs), ptr(ci.inv_norm), ci.n_docs, ci.dim,
                                 ptr(ci.row_group), ptr(qe), ptr(b), b.shape[1], ptr(d), d.shape[1], float(alpha), k,
                                 ptr(ids), ptr(sc), ptr(s_b), ptr(s_c), None, _lib.stream_ptr(dev)), "br_fuse_linear")
    return ids, sc, s_b, s_c


def fuse_linear(bm25_model, cosine_index, queries, query_embeddings, bm25_ids, dense_ids, k=10, alpha=0.5):
    """Linear fusion: f = alpha * n_b + (1 - alpha) * n_c over the union of the two lists, with n_b / n_c the exact BM25
    (as ``BM25.exact_scores``) and cosine (as ``CosineIndex.rerank``, or ``rerank_groups`` for an index with row_group)
    min-max-normalised per query over the union; a doc without sentence rows has n_c = 0.  -> (ids int32[Q, k],
    scores float64[Q, k], bm25 float64[Q, k], cos float32[Q, k] (NaN: no rows)) on the device.  alpha outside [0, 1] or
    an id outside [-1, corpus_size) raises BRError."""
    q_terms, q_off = bm25_model._to_device(*bm25_model.pack_queries(queries))
    return _fuse_linear_packed(bm25_model, cosine_index, q_terms, q_off, query_embeddings, bm25_ids, dense_ids, k, alpha)


def hybrid_search(bm25_model, cosine_index, queries, query_embeddings, k=10, n_bm25=100, n_dense=100, fusion="rrf",
                  rrf_c=60.0, weights=(1.0, 1.0), alpha=0.5, doc_filter=None, query_filter=None):
    """BM25 top-``n_bm25`` (docs with at least one matching term) and dense top-``n_dense`` (``CosineIndex.topk``, or
    ``topk_groups`` for an index with row_group whose groups are the BM25 documents), fused by ``fusion`` = "rrf"
    (``fuse_rrf``) or "linear" (``fuse_linear``) -> (ids int32[Q, k] local doc ids, scores float64[Q, k]) on the device.
    ``doc_filter`` / ``query_filter`` (over the BM25 documents, as in ``retrieve_top_n_batch``) go to both first stages,
    so every fused doc is allowed."""
    if fusion not in ("rrf", "linear"):
        raise ValueError(f"fusion must be 'rrf' or 'linear', got {fusion!r}")
    if not 1 <= int(n_bm25) <= _lib.BR_MAX_K:
        raise ValueError(f"n_bm25 must be in [1, {_lib.BR_MAX_K}]")
    if not 1 <= int(n_dense) <= MAX_DENSE:
        raise ValueError(f"n_dense must be in [1, {MAX_DENSE}]")
    k = _check_k(k)
    _check_docs(bm25_model, cosine_index)
    n = bm25_model.corpus_size
    q_terms, q_off = bm25_model._to_device(*bm25_model.pack_queries(queries))
    if q_terms.numel() == 0:                    # a batch without terms: a non-null buffer (n_terms is an upper bound)
        q_terms = torch.zeros(1, dtype=torch.int32, device=q_terms.device)
    nq = q_off.numel() - 1
    qe = _bf16(query_embeddings, bm25_model._device)
    if qe.dim() != 2 or qe.shape[0] != nq:
        raise ValueError(f"query_embeddings must be [{nq}, d] (one row per query), got {tuple(qe.shape)}")
    if nq == 0:                                 # br_topk_batch wants output buffers even for an empty batch
        dev = bm25_model._device
        return (torch.empty((0, k), dtype=torch.int32, device=dev), torch.empty((0, k), dtype=torch.float64, device=dev))
    b, _ = bm25_model.retrieve_top_n_batch((q_terms, q_off), min(int(n_bm25), n), positive_only=True,
                                           doc_filter=doc_filter, query_filter=query_filter)
    if cosine_index.row_group is None:
        d, _ = cosine_index.topk(qe, min(int(n_dense), n), doc_filter=doc_filter, query_filter=query_filter)
        base = cosine_index.doc_base
    else:
        d, _ = cosine_index.topk_groups(qe, min(int(n_dense), n), doc_filter=doc_filter, query_filter=query_filter)
        base = cosine_index.group_base
    d = torch.where(d >= 0, d - base, -1)
    if fusion == "rrf":
        return fuse_rrf(b, d, n, k, rrf_c, weights)
    ids, sc, _, _ = _fuse_linear_packed(bm25_model, cosine_index, q_terms, q_off, qe, b, d, k, alpha)
    return ids, sc
