"""Dense cosine similarity / re-rank on bf16 embeddings - the L3' layer of the reference
(team_run1.py:269-295: ``e / (e.norm() + 1e-10)`` on both sides, ``torch.matmul``, ``torch.topk``) on
the B200: a bf16 tcgen05 GEMM with the L2-normalisation and the top-k filter fused into its epilogue
(brute force over all docs), and a gather kernel for per-query candidate lists (BM25 top-1000 ->
cosine top-10).  Host code here only moves tensors; all arithmetic is in libbr_b200.so."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import check, ptr


def _bf16(x, dev):
    t = torch.as_tensor(x)
    if t.dtype != torch.bfloat16:
        t = t.to(torch.bfloat16)
    return t.to(dev).contiguous()


def set_cosine_option(name, value):
    """br_set_cosine_option: process-wide test switch of the brute-force path: "kernel" (0 auto, 1 forces the
    2-CTA multicast kernel that serves d > 768; both return bit-identical results)."""
    check(_lib.load().br_set_cosine_option(name.encode(), int(value)), "br_set_cosine_option")


def _row_group(row_group, n_rows, n_groups, dev):
    """-> (int32 device copy of ``row_group``, n_groups).  Shape, dtype and int32 range are checked here; the layout
    itself (non-decreasing, values in [0, n_groups)) is checked by the library on every grouped call."""
    rg = torch.as_tensor(row_group)
    if rg.dim() != 1 or rg.shape[0] != n_rows:
        raise ValueError(f"row_group must have shape [{n_rows}] (one group id per embedding row), got {tuple(rg.shape)}")
    if rg.dtype.is_floating_point or rg.dtype == torch.bool:
        raise ValueError(f"row_group must be an integer array, got {rg.dtype}")
    rg = rg.to(dev)
    lo, hi = (int(rg.min()), int(rg.max())) if n_rows else (0, -1)
    if lo < -2 ** 31 or hi >= 2 ** 31 - 1:
        raise ValueError("row_group values must fit int32")
    n_groups = hi + 1 if n_groups is None else int(n_groups)
    if not 1 <= n_groups < 2 ** 31:
        raise ValueError(f"n_groups must be in [1, 2^31), got {n_groups}")
    return rg.to(torch.int32).contiguous(), n_groups


class CosineIndex:
    """Doc embeddings resident in HBM with their inverse norms (``1/(||e||+1e-10)``, computed once).

    ``row_group`` (optional, int [n]): the group (document) of every row, non-decreasing - e.g. ``sentence_to_doc`` of a
    sentence-level index, whose rows are a document's sentences in order.  It enables ``topk_groups``.  ``n_groups``
    defaults to ``max(row_group) + 1``; pass the document count to include trailing documents without rows (filters over
    groups have that width).  ``group_base`` (default ``doc_base``) is added to the group ids ``topk_groups`` returns."""

    def __init__(self, doc_embeddings, device=None, doc_base=0, row_group=None, n_groups=None, group_base=None):
        lib = _lib.load()
        dev = _lib.require_cuda(device)
        self.device, self.doc_base = dev, int(doc_base)
        self.docs = _bf16(doc_embeddings, dev)
        if self.docs.dim() != 2 or self.docs.shape[1] % 8:
            raise ValueError("embeddings must be [n, d] with d a multiple of 8")
        self.n_docs, self.dim = self.docs.shape
        self.row_group, self.n_groups = None, None
        self.group_base = self.doc_base if group_base is None else int(group_base)
        if row_group is not None:
            self.row_group, self.n_groups = _row_group(row_group, self.n_docs, n_groups, dev)
        elif n_groups is not None:
            raise ValueError("n_groups needs row_group")
        with torch.cuda.device(dev):
            self.inv_norm = torch.empty(self.n_docs, dtype=torch.float32, device=dev)
            check(lib.br_row_inv_norms(ptr(self.docs), self.n_docs, self.dim, ptr(self.inv_norm), _lib.stream_ptr(dev)),
                  "br_row_inv_norms")

    def topk(self, query_embeddings, k=10, doc_filter=None, query_filter=None):
        """Brute-force cosine top-k -> (ids int64[Q, k] (doc_base + row), sims float32[Q, k]) on the device.
        ``doc_filter`` restricts the rows a query may return: bool [n] for the whole batch, or bool [F, n] with
        ``query_filter`` int [Q] (row of each query, -1 = unfiltered); exact, -1 pads when fewer than k rows are allowed."""
        lib = _lib.load()
        q = _bf16(query_embeddings, self.device)
        nq = q.shape[0]
        with torch.cuda.device(self.device):
            filt, _keep = _lib.pack_doc_filter(doc_filter, query_filter, nq, self.n_docs, self.device)
            ids = torch.empty((nq, k), dtype=torch.int64, device=self.device)
            sims = torch.empty((nq, k), dtype=torch.float32, device=self.device)
            check(lib.br_cosine_topk_filtered(ptr(self.docs), ptr(self.inv_norm), self.n_docs, self.dim, ptr(q), nq, int(k),
                                              self.doc_base, ptr(ids), ptr(sims), None if filt is None else C.byref(filt),
                                              _lib.stream_ptr(self.device)), "br_cosine_topk_filtered")
        return ids, sims

    def topk_groups(self, query_embeddings, k=10, doc_filter=None, query_filter=None):
        """Exact group-level top-k ("max-sim"): a group scores the best cosine of its rows (each computed as ``topk``
        computes it) -> (ids int64[Q, k] (group_base + group id), sims float32[Q, k]), ordered by (score desc, group id
        asc); groups without rows are never returned, -1 pads when fewer than k groups qualify.  ``doc_filter`` is over
        GROUP ids: bool [G] for the whole batch, or bool [F, G] with ``query_filter`` int [Q] (-1 = unfiltered)."""
        if self.row_group is None:
            raise ValueError("topk_groups needs an index built with row_group")
        lib = _lib.load()
        q = _bf16(query_embeddings, self.device)
        nq = q.shape[0]
        with torch.cuda.device(self.device):
            filt, _keep = _lib.pack_doc_filter(doc_filter, query_filter, nq, self.n_groups, self.device)
            ids = torch.empty((nq, k), dtype=torch.int64, device=self.device)
            sims = torch.empty((nq, k), dtype=torch.float32, device=self.device)
            check(lib.br_cosine_topk_grouped(ptr(self.docs), ptr(self.inv_norm), self.n_docs, self.dim, ptr(self.row_group),
                                             self.n_groups, ptr(q), nq, int(k), self.group_base, ptr(ids), ptr(sims),
                                             None if filt is None else C.byref(filt), _lib.stream_ptr(self.device)),
                  "br_cosine_topk_grouped")
        return ids, sims

    def rerank(self, query_embeddings, candidate_ids, k=10):
        """Cosine re-rank of per-query candidates [Q, c] (local rows, -1 = empty) -> (ids int32[Q, k], sims).  Any other
        id outside [0, n) raises BRError."""
        lib = _lib.load()
        q = _bf16(query_embeddings, self.device)
        cand = torch.as_tensor(candidate_ids).to(device=self.device, dtype=torch.int32).contiguous()
        nq, c = cand.shape
        with torch.cuda.device(self.device):
            ids = torch.empty((nq, k), dtype=torch.int32, device=self.device)
            sims = torch.empty((nq, k), dtype=torch.float32, device=self.device)
            check(lib.br_cosine_rerank(ptr(self.docs), ptr(self.inv_norm), self.n_docs, self.dim, ptr(q), nq, ptr(cand), c,
                                       int(k), ptr(ids), ptr(sims), _lib.stream_ptr(self.device)), "br_cosine_rerank")
        return ids, sims

    def rerank_groups(self, query_embeddings, candidate_groups, k=10):
        """Grouped re-rank of per-query candidate groups [Q, c] (local group ids, -1 = empty) -> (ids int32[Q, k] local
        group ids, sims float32[Q, k]).  A group scores the best cosine of its rows, each computed as ``rerank`` computes
        it; order (score desc, group id asc); a repeated group comes back once, groups without rows never, -1 / 0 pad.
        Any other id outside [0, n_groups) raises BRError."""
        if self.row_group is None:
            raise ValueError("rerank_groups needs an index built with row_group")
        lib = _lib.load()
        q = _bf16(query_embeddings, self.device)
        cand = torch.as_tensor(candidate_groups).to(device=self.device, dtype=torch.int32).contiguous()
        nq, c = cand.shape
        with torch.cuda.device(self.device):
            ids = torch.empty((nq, k), dtype=torch.int32, device=self.device)
            sims = torch.empty((nq, k), dtype=torch.float32, device=self.device)
            check(lib.br_cosine_rerank_grouped(ptr(self.docs), ptr(self.inv_norm), self.n_docs, self.dim, ptr(self.row_group),
                                               self.n_groups, ptr(q), nq, ptr(cand), c, int(k), ptr(ids), ptr(sims),
                                               _lib.stream_ptr(self.device)), "br_cosine_rerank_grouped")
        return ids, sims


def rerank_bm25_with_cosine(bm25_model, cosine_index, queries, query_embeddings, n_candidates=1000, k=10):
    """BASELINE config 3: BM25 top-``n_candidates`` then cosine re-rank to top-``k`` (the intended
    BM25 -> embedding re-rank of the reference, README.md:93-94; candidate cap 1000,
    text_preprocessing_and_embedding_setup.py:342)."""
    cand, _ = bm25_model.retrieve_top_n_batch(queries, min(n_candidates, bm25_model.corpus_size))
    return cosine_index.rerank(query_embeddings, cand, k)


def rerank_bm25_with_sentences(bm25_model, cosine_index, queries, query_embeddings, n_candidates=1000, k=10):
    """Config 3 at sentence granularity: BM25 top-``n_candidates`` documents, then each document scored by the best
    cosine of its sentence embeddings (``CosineIndex.rerank_groups`` over a sentence-level index whose groups are the
    BM25 documents) -> (document ids int32[Q, k], sims float32[Q, k])."""
    if cosine_index.n_groups != bm25_model.corpus_size:
        raise ValueError(f"the cosine index has {cosine_index.n_groups} groups, the BM25 model {bm25_model.corpus_size} "
                         "documents: the groups must be the BM25 documents")
    cand, _ = bm25_model.retrieve_top_n_batch(queries, min(n_candidates, bm25_model.corpus_size))
    return cosine_index.rerank_groups(query_embeddings, cand, k)
