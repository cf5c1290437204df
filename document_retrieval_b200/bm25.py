"""``BM25`` - the reference's per-language model object, backed by the B200 index.

Mirrors the class in bm25_ranking.ipynb:166-213 (``BM25(tokenized_corpus, k1, b)``,
``get_scores``, ``retrieve_top_n``) and its final_implementation.py:91-154 variant (no-arg
constructor + ``build(tokenized_corpus, lang)``, ``calculate_scores``, ``doc_lengths``,
``precomputed_idf``).  Scoring, selection and the index build run in libbr_b200.so (CUDA, sm_100a);
this file only converts between the reference's Python types and device buffers.

Added on top of the reference surface (SURVEY 8b): ``from_token_ids`` (int32 term ids instead of
strings), ``retrieve_top_n_batch`` / ``get_scores_batch`` (whole batches, torch CUDA tensors),
``variant`` / ``dedup_query`` (the three BM25 formulas in the reference, SURVEY appendix A),
``get_top_n`` as an alias of ``retrieve_top_n``, ``add_documents`` / ``add_texts`` / ``add_token_ids`` (grow a
built or loaded index, bit-identical to rebuilding the whole corpus) and ``remove_documents`` (shrink it, bit-identical
to rebuilding the kept documents).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import BRError, VARIANT_ID, check, ptr


def _as_i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


class BM25:
    def __init__(self, tokenized_corpus=None, k1=1.5, b=0.75, *, variant="notebook", dedup_query=None,
                 device=None):
        if variant not in VARIANT_ID:
            raise ValueError(f"variant must be one of {tuple(VARIANT_ID)}")
        self.k1 = k1
        self.b = b
        self.variant = variant
        # set(query) in the notebook class (bm25_ranking.ipynb:193); duplicates count in
        # score_documents_for_query (team_run1.py:183)
        self.dedup_query = (variant == "notebook") if dedup_query is None else bool(dedup_query)
        self._device = device
        self._h = None                 # br_index*
        self._vocab = None             # str -> term id (string API only; lazy when built from texts)
        self._terms = None             # term id -> str
        self._term_pool = None         # (offsets, utf-8 pool) of a loaded index file, decoded lazily
        self.vocabulary = None         # ingest.Vocabulary (GPU hash table) when built with from_texts
        self.bigrams = False           # from_texts(bigrams=True): query texts get the same 2-gram expansion
        self.vocab_size = 0
        self.corpus_size = 0
        self.avgdl = 0.0
        self.doc_base = 0
        self._csr = None               # cached host export
        self._df_idf = None
        if tokenized_corpus is not None:
            self.build(tokenized_corpus)

    # ------------------------------------------------------------------ build
    def build(self, tokenized_corpus, lang=None):
        """BM25.build (bm25_ranking.ipynb:178-189; final_implementation.py:105-118 takes an unused
        ``lang``).  ``tokenized_corpus`` is ``list[list[str]]``."""
        import pandas as pd
        n_docs = len(tokenized_corpus)
        if n_docs == 0:
            raise ZeroDivisionError("division by zero")            # sum(...)/corpus_size, :171
        lens = np.fromiter((len(d) for d in tokenized_corpus), dtype=np.int64, count=n_docs)
        doc_offsets = np.zeros(n_docs + 1, dtype=np.int64)
        np.cumsum(lens, out=doc_offsets[1:])
        flat = [w for d in tokenized_corpus for w in d]
        codes, uniques = pd.factorize(np.asarray(flat, dtype=object)) if flat else (np.zeros(0, np.int64), [])
        self.terms = [str(u) for u in uniques]
        self.vocabulary = None
        self._build_ids(doc_offsets, codes.astype(np.int32), max(len(self.terms), 1))
        return self

    # term strings: plain attributes for build(list[list[str]]), decoded lazily from the GPU vocabulary's
    # byte pool for from_texts (only the dict-valued attributes and list[str] queries need them)
    @property
    def terms(self):
        if self._terms is None and self.vocabulary is not None:
            self._terms = self.vocabulary.terms
        if self._terms is None and getattr(self, "_term_pool", None) is not None:
            off, pool = self._term_pool                     # loaded index file: decode on first use
            raw, o = pool.tobytes(), off.tolist()
            self._terms = [raw[o[i]:o[i + 1]].decode("utf-8") for i in range(len(o) - 1)]
        return self._terms

    @terms.setter
    def terms(self, v):
        self._terms, self._vocab, self._term_pool = v, None, None

    @property
    def vocab(self):
        if self._vocab is None and self.terms is not None:
            self._vocab = {w: i for i, w in enumerate(self.terms)}
        return self._vocab

    @vocab.setter
    def vocab(self, v):
        self._vocab = v

    @classmethod
    def from_texts(cls, texts, k1=1.5, b=0.75, *, bigrams=False, variant="notebook", dedup_query=None, device=None):
        """Build from preprocessed text instead of token lists: ``BM25([t.split() for t in texts])``
        (bm25_ranking.ipynb:299,306) with the tokenisation, the first-seen vocabulary and - with
        ``bigrams=True`` - the 2-gram expansion of bm25_ranking.ipynb:105-107 done on the GPU
        (ingest.py / csrc/br_ingest.cu).  Query with ``retrieve_top_n_texts`` (texts) or the usual
        token-list calls."""
        from .ingest import Vocabulary
        self = cls(None, k1, b, variant=variant, dedup_query=dedup_query, device=device)
        voc, doc_off, ids = Vocabulary.from_texts(texts, bigrams=bigrams, device=device)
        self.vocabulary = voc
        self.bigrams = bool(bigrams)
        self._device = voc.device
        self._build_ids(doc_off, ids, max(len(voc), 1))
        return self

    def retrieve_top_n_texts(self, query_texts, n=10, **kw):
        """``retrieve_top_n_batch([q.split() for q in query_texts], n)`` with the queries tokenised and
        looked up on the GPU (bm25_ranking.ipynb:341-347: ``tokenized_query = preprocessed_query.split()``)."""
        if self.vocabulary is None:
            from .ingest import Vocabulary
            if self.terms is None:
                raise BRError("retrieve_top_n_texts needs a model with a string vocabulary")
            self.vocabulary = Vocabulary.from_terms(self.terms, bigrams=self.bigrams, device=self._device)
        q_terms, q_off = self.vocabulary.encode_texts(query_texts)
        return self.retrieve_top_n_batch((q_terms, q_off), n, **kw)

    @classmethod
    def from_token_ids(cls, doc_offsets, token_ids, vocab_size, k1=1.5, b=0.75, *, variant="notebook",
                       dedup_query=None, device=None, doc_base=0, finalize=True):
        """Build from int32 term ids: ``doc_offsets`` int64[N+1], ``token_ids`` int32[T] (numpy or
        torch, host or device).  ``finalize=False`` stops after phase 1 so that a doc-sharded caller
        can all-reduce the statistics (see sharded.py)."""
        self = cls(None, k1, b, variant=variant, dedup_query=dedup_query, device=device)
        self._build_ids(doc_offsets, token_ids, int(vocab_size), doc_base=doc_base, finalize=finalize)
        return self

    def _build_ids(self, doc_offsets, token_ids, vocab_size, doc_base=0, finalize=True):
        lib = _lib.load()
        dev = _lib.require_cuda(self._device)
        self._device = dev
        with torch.cuda.device(dev):
            d_off = torch.as_tensor(doc_offsets).to(device=dev, dtype=torch.int64).contiguous()
            d_tok = torch.as_tensor(token_ids).to(device=dev, dtype=torch.int32).contiguous()
            n_docs = d_off.numel() - 1
            if n_docs <= 0:
                raise ZeroDivisionError("division by zero")
            h = C.c_void_p()
            check(lib.br_index_build(ptr(d_tok), ptr(d_off), n_docs, vocab_size, int(doc_base),
                                     _lib.stream_ptr(dev), C.byref(h)), "br_index_build")
        self._h = h
        self.vocab_size = vocab_size
        self.corpus_size = n_docs
        self.doc_base = int(doc_base)
        self._csr = self._df_idf = None
        if finalize:
            self.finalize()

    def finalize(self, n_stat=0, sum_dl_stat=0, df_stat=None):
        """Phase 2: fix N / avgdl / df (global statistics for a doc shard) and compute the weights."""
        lib = _lib.load()
        df_arr = None if df_stat is None else np.ascontiguousarray(df_stat, dtype=np.int64)
        with torch.cuda.device(self._device):
            check(lib.br_index_finalize(self._h, float(self.k1), float(self.b), VARIANT_ID[self.variant],
                                        float(n_stat), float(sum_dl_stat),
                                        None if df_arr is None else df_arr.ctypes.data,
                                        _lib.stream_ptr(self._device)), "br_index_finalize")
        st = self.stats()
        self.avgdl = st["avgdl"]
        self._df_idf = None
        return self

    # ------------------------------------------------------------------ append
    # Each add_* is the append counterpart of one constructor: the new docs get ids corpus_size .., and the index is
    # re-finalised with this model's k1 / b / variant, bit-identical to building the concatenated corpus from scratch.
    def add_documents(self, tokenized_corpus):
        """Append token lists (``list[list[str]]``, as for ``BM25(...)`` / ``build``).  New term strings are appended to
        ``terms`` in first-seen order.  Returns ``self``."""
        if self.bigrams:
            raise ValueError("add_documents: this model expands its texts with bigrams, which token lists would skip; "
                             "use add_texts")
        if len(tokenized_corpus) == 0:
            return self
        self._check_mutable()
        terms = self.terms
        if terms is None:
            raise ValueError("add_documents needs a model with a string vocabulary (use add_token_ids)")
        import pandas as pd
        n_docs = len(tokenized_corpus)
        lens = np.fromiter((len(d) for d in tokenized_corpus), dtype=np.int64, count=n_docs)
        doc_offsets = np.zeros(n_docs + 1, dtype=np.int64)
        np.cumsum(lens, out=doc_offsets[1:])
        flat = [w for d in tokenized_corpus for w in d]
        codes, uniques = pd.factorize(np.asarray(flat, dtype=object)) if flat else (np.zeros(0, np.int64), [])
        vocab, new_terms = self.vocab, []
        ids_of_unique = np.empty(len(uniques), dtype=np.int32)
        for i, u in enumerate(uniques):
            t = vocab.get(str(u))
            if t is None:
                t = len(terms) + len(new_terms)
                new_terms.append(str(u))
            ids_of_unique[i] = t
        grown = terms + new_terms
        self._append_ids(doc_offsets, ids_of_unique[codes], max(len(grown), self.vocab_size))
        if new_terms:
            self.vocabulary = None     # a GPU vocabulary lacks the new terms: retrieve_top_n_texts rebuilds it from terms
            self.terms = grown
        return self

    def add_texts(self, texts):
        """Append preprocessed texts (as for ``from_texts``), tokenised on the GPU; new terms are added to the GPU
        vocabulary (br_vocab_extend), with the model's 2-gram expansion when it has one.  A model with string terms but
        no GPU vocabulary (built by ``build``, loaded from a file, unpickled) first gets one from its terms.  Returns
        ``self``."""
        from .ingest import Vocabulary
        if not isinstance(texts, tuple) and len(texts) == 0:
            return self
        self._check_mutable()
        if self.vocabulary is None:
            if self.terms is None:
                raise BRError("add_texts needs a model with a string vocabulary")
            self.vocabulary = Vocabulary.from_terms(self.terms, bigrams=self.bigrams, device=self._device)
        voc = self.vocabulary
        n_terms = len(voc)
        doc_off, ids = voc.extend_texts(texts)
        try:
            self._append_ids(doc_off, ids, max(len(voc), self.vocab_size))
        except Exception:
            voc._truncate(n_terms)     # the index refused the documents: their new terms leave the vocabulary too
            raise
        self.terms = None              # decoded again from the grown vocabulary
        return self

    def add_token_ids(self, doc_offsets, token_ids, vocab_size=None):
        """Append int32 term ids (as for ``from_token_ids``): ``doc_offsets`` int64[n+1], ``token_ids`` int32[T], numpy or
        torch, host or device.  ``vocab_size`` (default: the current one) may grow the vocabulary of a model without
        term strings only.  Returns ``self``."""
        vocab_size = self.vocab_size if vocab_size is None else int(vocab_size)
        if vocab_size > self.vocab_size and self.terms is not None:
            raise ValueError("add_token_ids cannot add terms without strings to a model with a string vocabulary "
                             "(use add_documents or add_texts)")
        if len(doc_offsets) <= 1:
            return self
        self._check_mutable()
        self._append_ids(doc_offsets, token_ids, vocab_size)
        return self

    def _check_mutable(self):
        """A doc shard is finalised with global statistics; re-finalising it with its local ones would silently break
        it, so documents are only added to or removed from it through a sharded wrapper."""
        self._require()
        lib = _lib.load()
        n_stat, sum_dl_stat = C.c_double(), C.c_double()
        check(lib.br_index_stats_in_force(self._h, C.byref(n_stat), C.byref(sum_dl_stat)), "br_index_stats_in_force")
        st = self.stats()
        df, _ = self._export_df_idf()
        if (n_stat.value != st["n_docs"] or sum_dl_stat.value != st["sum_dl"]
                or not np.array_equal(df, self.local_df_tensor().cpu().numpy())):
            raise BRError("this index is a doc shard finalised with global statistics: documents cannot be added to or "
                          "removed from it alone")

    def _append_ids(self, doc_offsets, token_ids, vocab_size):
        lib = _lib.load()
        dev = self._device
        with torch.cuda.device(dev):
            d_off = torch.as_tensor(doc_offsets).to(device=dev, dtype=torch.int64).contiguous()
            d_tok = torch.as_tensor(token_ids).to(device=dev, dtype=torch.int32).contiguous()
            n_docs = d_off.numel() - 1
            if n_docs <= 0:
                return
            if d_tok.numel() == 0:
                d_tok = torch.zeros(1, dtype=torch.int32, device=dev)      # only empty docs: nothing is read
            check(lib.br_index_append(self._h, ptr(d_tok), ptr(d_off), n_docs, int(vocab_size), _lib.stream_ptr(dev)),
                  "br_index_append")
        self.vocab_size = int(vocab_size)
        self.corpus_size += n_docs
        self._csr = None
        self.finalize()

    # ------------------------------------------------------------------ remove
    def remove_documents(self, docs):
        """Remove documents: ``docs`` is a bool mask [N] (True = remove) or integer local doc ids (duplicates count
        once), numpy or torch, host or device.  Returns ``self``.

        The kept docs keep their order and are renumbered by rank: with ``kept = np.flatnonzero(~mask)``, new id ``i`` is
        old id ``kept[i]`` (update a ``doc_id_maps`` list with ``[old_map[d] for d in kept]``).  ``doc_base``, the term
        ids, ``vocab_size``, ``terms`` and the GPU vocabulary do not change; a term left in no doc keeps its id with
        df 0 and drops out of the ``df`` / ``idf`` / ``inverted_index`` dicts.  The index is re-finalised with this
        model's k1 / b / variant and equals, bit for bit, the index built from scratch from the kept docs over the same
        vocabulary.  Removing nothing is a no-op; removing every doc is refused (ValueError).

        A ``CosineIndex`` holding the same docs is not changed: rebuild it from the kept rows (``emb[kept]``; for a
        grouped index the kept rows with ``row_group`` remapped by the same rank), which is exact because a row's norm
        depends on that row only."""
        self._require()
        N = self.corpus_size
        if isinstance(docs, (list, tuple)):
            if len(docs) == 0:
                return self
            docs = np.asarray(docs)
        t = torch.as_tensor(docs)
        if t.dtype == torch.bool:
            if tuple(t.shape) != (N,):
                raise ValueError(f"remove_documents: a mask must have shape [{N}], got {list(t.shape)}")
        elif t.is_floating_point() or t.is_complex():
            raise ValueError(f"remove_documents: docs must be a bool mask or integer doc ids, got {t.dtype}")
        else:
            t = t.reshape(-1)
            if t.numel() == 0:
                return self
            lo, hi = int(t.min()), int(t.max())
            if lo < 0 or hi >= N:
                raise ValueError(f"remove_documents: doc ids must be in [0, {N}), got [{lo}, {hi}]")
        dev = self._device
        with torch.cuda.device(dev):
            if t.dtype == torch.bool:
                mask = t.to(device=dev, dtype=torch.uint8).contiguous()
            else:
                mask = torch.zeros(N, dtype=torch.uint8, device=dev)
                mask[t.to(device=dev, dtype=torch.int64)] = 1
            n_removed = int(mask.sum())
        if n_removed == 0:
            return self
        if n_removed == N:
            raise ValueError("remove_documents: every document would be removed; an index holds at least one")
        self._check_mutable()
        self._remove_mask(mask, n_removed)
        return self

    def _remove_mask(self, mask, n_removed):
        dev = self._device
        with torch.cuda.device(dev):
            check(_lib.load().br_index_remove(self._h, ptr(mask), _lib.stream_ptr(dev)), "br_index_remove")
        self.corpus_size -= n_removed
        self._csr = None
        self.finalize()

    def stats(self):
        lib = _lib.load()
        n, v, nnz, avg, sdl, base = (C.c_int64(), C.c_int32(), C.c_int64(), C.c_double(), C.c_int64(), C.c_int64())
        check(lib.br_index_stats(self._h, C.byref(n), C.byref(v), C.byref(nnz), C.byref(avg), C.byref(sdl),
                                 C.byref(base)), "br_index_stats")
        return dict(n_docs=n.value, vocab=v.value, nnz=nnz.value, avgdl=avg.value, sum_dl=sdl.value,
                    doc_base=base.value)

    def local_df_tensor(self):
        """uint32[V] shard-local df on the device, as an int32 torch view (for the all-reduce)."""
        lib = _lib.load()
        p = lib.br_index_df_dev(self._h)
        n = self.vocab_size

        class _Arr:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (p, False), "version": 3}
        return torch.as_tensor(_Arr(), device=self._device)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().br_index_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ queries
    def _require(self):
        if self._h is None:
            raise BRError("BM25 index not built (call build()/from_token_ids first)")

    def _encode(self, query):
        """One query -> int32 term ids (unknown strings -> -1, which the kernels skip like
        ``if word not in self.idf: continue``, bm25_ranking.ipynb:195-196)."""
        if isinstance(query, np.ndarray) and query.dtype.kind in "iu":
            return query.astype(np.int32)
        if torch.is_tensor(query):
            return query.detach().cpu().numpy().astype(np.int32)
        out = np.empty(len(query), dtype=np.int32)
        for i, w in enumerate(query):
            if isinstance(w, (int, np.integer)) and self.vocab is None:
                out[i] = int(w)
            else:
                out[i] = -1 if self.vocab is None else self.vocab.get(w, -1)
        return out

    def pack_queries(self, queries):
        """list of token lists | (q_terms, q_offsets) -> pinned host (q_terms int32, q_offsets int32)."""
        if isinstance(queries, tuple) and len(queries) == 2 and all(
                isinstance(x, np.ndarray) or torch.is_tensor(x) for x in queries):
            # packed form: (q_terms, q_offsets) ARRAYS with q_offsets[0] == 0 and q_offsets[-1] == len(q_terms); a tuple of
            # two token lists is a batch of two queries, not this
            q_terms = torch.as_tensor(queries[0]).to(torch.int32).contiguous()
            q_off = torch.as_tensor(queries[1]).to(torch.int32).contiguous()
            if q_off.numel() < 1 or q_terms.dim() != 1 or q_off.dim() != 1:
                raise ValueError("packed queries: q_terms and q_offsets must be 1-D and q_offsets non-empty")
            if q_off.device.type == "cpu" and (int(q_off[0]) != 0 or int(q_off[-1]) != q_terms.numel()):
                raise ValueError("packed queries: q_offsets must start at 0 and end at len(q_terms)")
            return q_terms, q_off
        enc = [self._encode(q) for q in queries]
        lens = np.fromiter((e.size for e in enc), dtype=np.int64, count=len(enc))
        q_off = np.zeros(len(enc) + 1, dtype=np.int32)
        np.cumsum(lens, out=q_off[1:])
        q_terms = np.concatenate(enc).astype(np.int32) if enc and q_off[-1] > 0 else np.zeros(0, np.int32)
        return torch.from_numpy(q_terms), torch.from_numpy(q_off)

    def _to_device(self, q_terms, q_off):
        dev = self._device
        if q_terms.device != dev:
            if q_terms.numel() == 0:
                q_terms = torch.zeros(1, dtype=torch.int32)
            q_terms = q_terms.pin_memory().to(dev, non_blocking=True) if q_terms.device.type == "cpu" else q_terms.to(dev)
        if q_off.device != dev:
            q_off = q_off.pin_memory().to(dev, non_blocking=True) if q_off.device.type == "cpu" else q_off.to(dev)
        return q_terms, q_off

    def get_scores_batch(self, queries):
        """fp32[Q, N] scores on the device (batched get_scores; small N / debugging)."""
        self._require()
        lib = _lib.load()
        q_terms, q_off = self._to_device(*self.pack_queries(queries))
        nq = q_off.numel() - 1
        with torch.cuda.device(self._device):
            out = torch.empty((nq, self.corpus_size), dtype=torch.float32, device=self._device)
            check(lib.br_score_batch(self._h, ptr(q_terms), ptr(q_off), nq, int(self.dedup_query), ptr(out),
                                     _lib.stream_ptr(self._device)), "br_score_batch")
        return out

    def get_scores(self, query):
        """bm25_ranking.ipynb:191-204 -> np.ndarray[float64, (N,)] (fp32 accumulation widened; the
        error bound of br_score_batch in include/br_b200.h)."""
        return self.get_scores_batch([query])[0].double().cpu().numpy()

    calculate_scores = get_scores          # final_implementation.py:127

    def retrieve_top_n_batch(self, queries, n=10, positive_only=False, return_counts=False, doc_filter=None,
                             query_filter=None):
        """Batched retrieve_top_n -> (ids int32[Q, n] local doc ids (-1 pads), scores float64[Q, n])
        as CUDA tensors, ordered by (float64 score desc, doc id asc).

        ``doc_filter`` restricts what may be returned: a bool [N] allow-list for the whole batch, or bool [F, N] rows
        with ``query_filter`` int [Q] (the row of each query, -1 = unfiltered).  A filtered query's result is the
        result over its allowed docs only - same scores (N, avgdl and idf stay those of the whole index), -1 padding
        when fewer than n docs are allowed."""
        self._require()
        lib = _lib.load()
        n = int(n)
        if not 1 <= n <= _lib.BR_MAX_K:
            raise ValueError(f"n must be in [1, {_lib.BR_MAX_K}] for the batched call")
        q_terms, q_off = self._to_device(*self.pack_queries(queries))
        nq = q_off.numel() - 1
        dev = self._device
        with torch.cuda.device(dev):
            filt, _keep = _lib.pack_doc_filter(doc_filter, query_filter, nq, self.corpus_size, dev)
            ids = torch.empty((nq, n), dtype=torch.int32, device=dev)
            sc = torch.empty((nq, n), dtype=torch.float64, device=dev)
            cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
            check(lib.br_topk_batch_filtered(self._h, ptr(q_terms), ptr(q_off), nq, int(q_terms.numel()), n,
                                             int(self.dedup_query), int(positive_only), ptr(ids), ptr(sc), ptr(cnt),
                                             None if filt is None else C.byref(filt), _lib.stream_ptr(dev)),
                  "br_topk_batch_filtered")
        return (ids, sc, cnt) if return_counts else (ids, sc)

    def retrieve_records_batch(self, queries, n=10, positive_only=False, doc_filter=None, query_filter=None):
        """retrieve_top_n_batch as packed records int64[Q, n, 2]: [..., 0] = global doc id (doc_base + local id, -1
        pads), [..., 1] = the float64 score's bits - what a doc-sharded caller all-gathers in one collective.
        ``doc_filter`` / ``query_filter``: as in retrieve_top_n_batch (over this index's local doc ids)."""
        self._require()
        lib = _lib.load()
        n = int(n)
        if not 1 <= n <= _lib.BR_MAX_K:
            raise ValueError(f"n must be in [1, {_lib.BR_MAX_K}] for the batched call")
        q_terms, q_off = self._to_device(*self.pack_queries(queries))
        nq = q_off.numel() - 1
        dev = self._device
        with torch.cuda.device(dev):
            filt, _keep = _lib.pack_doc_filter(doc_filter, query_filter, nq, self.corpus_size, dev)
            rec = torch.empty((nq, n, 2), dtype=torch.int64, device=dev)
            check(lib.br_topk_batch_records_filtered(self._h, ptr(q_terms), ptr(q_off), nq, int(q_terms.numel()), n,
                                                     int(self.dedup_query), int(positive_only), ptr(rec), None,
                                                     None if filt is None else C.byref(filt), _lib.stream_ptr(dev)),
                  "br_topk_batch_records_filtered")
        return rec

    def exact_scores(self, query):
        """float64[N] exact re-evaluation of the reference formula for every doc (device tensor)."""
        self._require()
        lib = _lib.load()
        dev = self._device
        q_terms, q_off = self._to_device(*self.pack_queries([query]))
        with torch.cuda.device(dev):
            cand = torch.arange(self.corpus_size, dtype=torch.int32, device=dev)
            off = torch.tensor([0, self.corpus_size], dtype=torch.int64, device=dev)
            out = torch.empty(self.corpus_size, dtype=torch.float64, device=dev)
            check(lib.br_rescore_docs(self._h, ptr(q_terms), ptr(q_off), 1, int(self.dedup_query), ptr(cand),
                                      ptr(off), ptr(out), _lib.stream_ptr(dev)), "br_rescore_docs")
        return out

    def tfidf_cosine_top_n_batch(self, queries, n=200):
        """First stage of rank_documents_with_cosine_similarity_and_bm25
        (cosine_similarity_bm25_reranking.py:210-229): top-``n`` docs by sparse TF-IDF cosine ->
        (ids int32[Q, n], scores float64[Q, n] = cosine * ||q||) on the device."""
        self._require()
        lib = _lib.load()
        q_terms, q_off = self._to_device(*self.pack_queries(queries))
        nq = q_off.numel() - 1
        dev = self._device
        with torch.cuda.device(dev):
            ids = torch.empty((nq, n), dtype=torch.int32, device=dev)
            sc = torch.empty((nq, n), dtype=torch.float64, device=dev)
            check(lib.br_tfidf_cosine_topk(self._h, ptr(q_terms), ptr(q_off), nq, int(n), ptr(ids), ptr(sc), None,
                                           _lib.stream_ptr(dev)), "br_tfidf_cosine_topk")
        return ids, sc

    def rerank_scores_v3(self, queries, cand_ids):
        """bm25_score (cosine_similarity_bm25_reranking.py:185-195) of every (query, candidate) pair:
        ``cand_ids`` int32[Q, c] (local ids, -1 = empty) -> float64[Q, c] on the device."""
        self._require()
        lib = _lib.load()
        q_terms, q_off = self._to_device(*self.pack_queries(queries))
        nq = q_off.numel() - 1
        dev = self._device
        cand = torch.as_tensor(cand_ids).to(device=dev, dtype=torch.int32).contiguous()
        c = cand.shape[1]
        with torch.cuda.device(dev):
            off = torch.arange(nq + 1, dtype=torch.int64, device=dev) * c
            out = torch.empty((nq, c), dtype=torch.float64, device=dev)
            check(lib.br_rerank_v3_scores(self._h, ptr(q_terms), ptr(q_off), nq, ptr(cand), ptr(off), ptr(out),
                                          _lib.stream_ptr(dev)), "br_rerank_v3_scores")
        return out

    def retrieve_top_n(self, query, n=10, doc_filter=None):
        """bm25_ranking.ipynb:206-213 -> np.ndarray[int64] of local doc indices, best first.
        ``n >= N`` returns the full ranking (:208-209).  Ties: doc id ascending.  ``doc_filter`` (bool [N]): rank only
        the allowed docs (the result then holds at most as many ids as docs are allowed)."""
        self._require()
        n = int(n)
        N = self.corpus_size
        if doc_filter is not None:
            f = torch.as_tensor(doc_filter)
            if f.dtype != torch.bool or f.dim() != 1 or f.shape[0] != N:
                raise ValueError(f"doc_filter must be a bool array of shape [{N}]")
        if n >= N or n > _lib.BR_MAX_K:
            s = self.exact_scores(query)
            if doc_filter is None:
                order = torch.sort(-s, stable=True).indices[:min(n, N)]     # stable: ties keep id order
            else:
                allowed = torch.nonzero(f.to(s.device)).flatten()
                order = allowed[torch.sort(-s[allowed], stable=True).indices][:min(n, N)]
            return order.cpu().numpy().astype(np.int64)
        if n <= 0:
            return np.zeros(0, dtype=np.int64)
        if doc_filter is None:
            ids, _ = self.retrieve_top_n_batch([query], n)
            return ids[0].cpu().numpy().astype(np.int64)
        ids, _ = self.retrieve_top_n_batch([query], n, doc_filter=f)
        row = ids[0].cpu().numpy().astype(np.int64)
        return row[row >= 0]

    get_top_n = retrieve_top_n             # BASELINE.json's wording (rank_bm25 style)

    def set_profiling(self, on=True):
        check(_lib.load().br_set_profiling(self._h, int(bool(on))), "br_set_profiling")

    def set_option(self, name, value):
        """Library tuning / test switches: "fused" (0 = dense path only), "fused_long" (0 = no long-query tiled pass),
        "defer_pm" (MaxScore deferral budget, per mille of the threshold, 0-1000)."""
        check(_lib.load().br_set_option(self._h, name.encode(), int(value)), "br_set_option")

    def query_stats(self):
        st = _lib.QueryStats()
        check(_lib.load().br_last_query_stats(self._h, C.byref(st)), "br_last_query_stats")
        return {f: getattr(st, f) for f, _ in st._fields_}

    # ------------------------------------------------------------------ reference attributes
    def _export_csr(self):
        if self._csr is None:
            self._require()
            st = self.stats()
            row_ptr = np.empty(st["vocab"] + 1, np.int64)
            doc = np.empty(st["nnz"], np.int32)
            tf = np.empty(st["nnz"], np.int32)
            dl = np.empty(st["n_docs"], np.int32)
            with torch.cuda.device(self._device):
                check(_lib.load().br_index_export_csr(self._h, row_ptr.ctypes.data, doc.ctypes.data, tf.ctypes.data,
                                                      dl.ctypes.data), "br_index_export_csr")
            self._csr = dict(row_ptr=row_ptr, doc=doc, tf=tf, dl=dl)
        return self._csr

    def _export_df_idf(self):
        if self._df_idf is None:
            self._require()
            df = np.empty(self.vocab_size, np.int64)
            idf = np.empty(self.vocab_size, np.float64)
            check(_lib.load().br_index_export_df_idf(self._h, df.ctypes.data, idf.ctypes.data), "br_index_export_df_idf")
            self._df_idf = (df, idf)
        return self._df_idf

    def _key(self, t):
        return self.terms[t] if self.terms is not None else int(t)

    @property
    def df(self):
        """{term: document frequency} (bm25_ranking.ipynb:173,185)."""
        df, _ = self._export_df_idf()
        return {self._key(t): int(df[t]) for t in np.nonzero(df)[0]}

    @property
    def idf(self):
        """{term: idf} (bm25_ranking.ipynb:188-189)."""
        df, idf = self._export_df_idf()
        return {self._key(t): float(idf[t]) for t in np.nonzero(df)[0]}

    precomputed_idf = idf                  # final_implementation.py:124-125

    @property
    def inverted_index(self):
        """{term: [doc ids ascending]} (bm25_ranking.ipynb:175,186)."""
        c = self._export_csr()
        rp = c["row_ptr"]
        return {self._key(t): c["doc"][rp[t]:rp[t + 1]].tolist() for t in range(self.vocab_size) if rp[t + 1] > rp[t]}

    @property
    def term_freqs(self):
        """[{term: tf}] per doc (bm25_ranking.ipynb:176,180-183)."""
        c = self._export_csr()
        rp = c["row_ptr"]
        out = [dict() for _ in range(self.corpus_size)]
        for t in range(self.vocab_size):
            k = self._key(t)
            for d, f in zip(c["doc"][rp[t]:rp[t + 1]].tolist(), c["tf"][rp[t]:rp[t + 1]].tolist()):
                out[d][k] = f
        return out

    @property
    def doc_lengths(self):
        """{doc id: token count} (final_implementation.py:121-122)."""
        return dict(enumerate(self._export_csr()["dl"].tolist()))

    # ------------------------------------------------------------------ native (de)serialisation
    def save(self, path):
        """Flat binary index file: a JSON header followed by the raw arrays (row_ptr int64, doc int32, tf uint16,
        dl int32, optionally the statistics in force for a doc shard and the vocabulary as a UTF-8 byte pool + offsets),
        each at a 4096-byte aligned offset.  No pickle anywhere.  Replaces the joblib / pickle model files whose loading
        dominated the reference's run time (bm25_ranking.ipynb:222-251, final_implementation.py:187-287): ``load``
        streams the arrays through pinned memory to the GPU, validates them there and rebuilds the weights, skip tables
        and rows on the device."""
        from . import indexfile
        indexfile.save(self, path)

    @classmethod
    def load(cls, path, device=None):
        from . import indexfile
        return indexfile.load(cls, path, device)

    # ------------------------------------------------------------------ pickling (joblib.dump, :312)
    def __getstate__(self):
        st = dict(k1=self.k1, b=self.b, variant=self.variant, dedup_query=self.dedup_query, terms=self.terms,
                  vocab_size=self.vocab_size, corpus_size=self.corpus_size, doc_base=self.doc_base, csr=None,
                  stat=None, bigrams=self.bigrams)
        if self._h is not None:
            st["csr"] = self._export_csr()
            s = self.stats()
            df, _ = self._export_df_idf()
            st["stat"] = dict(avgdl=s["avgdl"], df=df)
        return st

    def __setstate__(self, st, device=None):
        self.__init__(None, st["k1"], st["b"], variant=st["variant"], dedup_query=st["dedup_query"], device=device)
        self.terms = st["terms"]
        self.bigrams = bool(st.get("bigrams", False))
        self.vocab_size, self.corpus_size, self.doc_base = st["vocab_size"], st["corpus_size"], st["doc_base"]
        c = st["csr"]
        if c is None:
            return
        lib = _lib.load()
        dev = _lib.require_cuda(self._device)
        self._device = dev
        h = C.c_void_p()
        with torch.cuda.device(dev):
            check(lib.br_index_import_csr(c["row_ptr"].ctypes.data, c["doc"].ctypes.data, c["tf"].ctypes.data,
                                          c["dl"].ctypes.data, self.corpus_size, self.vocab_size, self.doc_base,
                                          _lib.stream_ptr(dev), C.byref(h)), "br_index_import_csr")
        self._h = h
        self._csr = c
        # restore the statistics in force (they differ from the local ones for a doc shard)
        df = st["stat"]["df"]
        local_sum = int(c["dl"].sum())
        n_stat = 0 if np.array_equal(df, np.diff(c["row_ptr"])) else None
        if n_stat == 0:
            self.finalize()
        else:
            raise BRError("pickled doc shards must be re-finalised by the sharded wrapper")
        assert abs(self.avgdl - st["stat"]["avgdl"]) <= 1e-12 * max(1.0, self.avgdl), (local_sum, self.avgdl)
