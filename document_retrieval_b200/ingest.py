"""Text -> term ids on the GPU: the step right before the hot path (SURVEY 8f rank 2).

The reference tokenises a language's preprocessed corpus with ``[text.split() for text in lang_texts]``
(bm25_ranking.ipynb:299) and lets ``BM25.build`` grow its vocabulary through dict inserts, one per token
(bm25_ranking.ipynb:180-186); for fr/de/es/it the preprocessing also appends 2-grams
``tokens + ['_'.join(gram) for gram in ngrams(tokens, 2)]`` (bm25_ranking.ipynb:105-107).  Here the
texts cross PCIe once as one UTF-8 buffer (Arrow ``large_string`` layout, built by pyarrow in C) and
``libbr_b200.so`` does the rest: ``str.split()`` tokenisation, vocabulary in first-seen order, term ids
(csrc/br_ingest.cu).  Host code below only moves buffers; there is no CPU tokeniser behind it."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check, ptr


def pack_texts(texts):
    """list[str] (non-``str`` entries count as "", bm25_ranking.ipynb:85-86) -> host
    (uint8[n_bytes] UTF-8 of all texts back to back, int64[n+1] byte offsets)."""
    import pyarrow as pa
    if isinstance(texts, tuple) and len(texts) == 2:
        return np.ascontiguousarray(texts[0], dtype=np.uint8), np.ascontiguousarray(texts[1], dtype=np.int64)
    try:
        arr = pa.array(texts, type=pa.large_utf8())
        if arr.null_count:
            raise TypeError
    except (pa.ArrowInvalid, pa.ArrowTypeError, TypeError):
        arr = pa.array([t if isinstance(t, str) else "" for t in texts], type=pa.large_utf8())
    if isinstance(arr, pa.ChunkedArray):
        arr = arr.combine_chunks()
    n = len(arr)
    _, off_buf, data_buf = arr.buffers()
    off = np.frombuffer(off_buf, dtype=np.int64, count=n + 1, offset=arr.offset * 8) if n or off_buf else np.zeros(1, np.int64)
    data = np.frombuffer(data_buf, dtype=np.uint8) if data_buf is not None and data_buf.size else np.zeros(0, np.uint8)
    if off[0] != 0:
        data, off = data[off[0]:off[-1]], off - off[0]
    return np.ascontiguousarray(data[:off[-1]]), np.ascontiguousarray(off)


def _to_dev(a, dev, dtype):
    t = torch.from_numpy(a) if a.size else torch.zeros(1, dtype=dtype)
    return t.to(dev, non_blocking=False)


class Vocabulary:
    """term string <-> term id, resident on the GPU as a sorted 64-bit hash table plus the byte pool of
    the term strings (first occurrence of each term in the corpus)."""

    def __init__(self, handle, device, bigrams=False):
        self._h, self.device, self.bigrams = handle, device, bool(bigrams)
        self._terms = None

    # ------------------------------------------------------------------ build / encode
    @staticmethod
    def _tokenize_count(lib, dev, texts, bigrams):
        data, off = pack_texts(texts)
        n_docs = off.size - 1
        d_text, d_off = _to_dev(data, dev, torch.uint8), _to_dev(off, dev, torch.int64)
        tok_off = torch.empty(n_docs + 1, dtype=torch.int64, device=dev)
        n_tok = C.c_int64()
        check(lib.br_tokenize_count(ptr(d_text), ptr(d_off), n_docs, int(bigrams), ptr(tok_off), C.byref(n_tok),
                                    _lib.stream_ptr(dev)), "br_tokenize_count")
        return d_text, d_off, n_docs, tok_off, n_tok.value

    @classmethod
    def from_texts(cls, texts, bigrams=False, device=None):
        """-> (Vocabulary, doc_offsets int64[N+1], token_ids int32[T]) with the two arrays on the device,
        ready for ``BM25.from_token_ids``."""
        lib = _lib.load()
        dev = _lib.require_cuda(device)
        with torch.cuda.device(dev):
            d_text, d_off, n_docs, tok_off, n_tok = cls._tokenize_count(lib, dev, texts, bigrams)
            ids = torch.empty(max(n_tok, 1), dtype=torch.int32, device=dev)[:n_tok]
            h = C.c_void_p()
            check(lib.br_vocab_build(ptr(d_text), ptr(d_off), n_docs, int(bigrams), ptr(tok_off), n_tok, ptr(ids),
                                     _lib.stream_ptr(dev), C.byref(h)), "br_vocab_build")
        return cls(h, dev, bigrams), tok_off, ids

    def extend_texts(self, texts):
        """Grow the vocabulary with the terms of new documents -> (doc_offsets int64[N+1], token_ids int32[T]) on the
        device, like ``from_texts``.  Known terms keep their ids; new terms are numbered after the existing ones in order
        of first occurrence, so ``from_texts(A)`` extended with B equals ``from_texts(A + B)``."""
        lib = _lib.load()
        dev = self.device
        with torch.cuda.device(dev):
            d_text, d_off, n_docs, tok_off, n_tok = self._tokenize_count(lib, dev, texts, self.bigrams)
            ids = torch.empty(max(n_tok, 1), dtype=torch.int32, device=dev)[:n_tok]
            check(lib.br_vocab_extend(self._h, ptr(d_text), ptr(d_off), n_docs, int(self.bigrams), ptr(tok_off), n_tok,
                                      ptr(ids), _lib.stream_ptr(dev)), "br_vocab_extend")
        self._terms = None
        return tok_off, ids

    def _truncate(self, n_terms):
        """Keep the first ``n_terms`` terms (takes back an ``extend_texts`` whose documents an index refused)."""
        off, pool = self._export()
        old = self._h
        self.__setstate__(dict(pool_off=off[:n_terms + 1], pool=pool[:off[n_terms]], bigrams=self.bigrams))
        _lib.load().br_vocab_destroy(old)

    def encode_texts(self, texts):
        """Query texts -> (q_terms int32[T], q_offsets int64[Q+1]) on the device; -1 = out of vocabulary."""
        lib = _lib.load()
        dev = self.device
        with torch.cuda.device(dev):
            d_text, d_off, n, tok_off, n_tok = self._tokenize_count(lib, dev, texts, self.bigrams)
            ids = torch.empty(max(n_tok, 1), dtype=torch.int32, device=dev)[:n_tok]
            check(lib.br_vocab_lookup(self._h, ptr(d_text), ptr(d_off), n, int(self.bigrams), ptr(tok_off), n_tok,
                                      ptr(ids), _lib.stream_ptr(dev)), "br_vocab_lookup")
        return ids, tok_off

    # ------------------------------------------------------------------ strings
    def __len__(self):
        n = C.c_int64()
        check(_lib.load().br_vocab_stats(self._h, C.byref(n), None), "br_vocab_stats")
        return n.value

    def _export(self):
        n, nb = C.c_int64(), C.c_int64()
        lib = _lib.load()
        check(lib.br_vocab_stats(self._h, C.byref(n), C.byref(nb)), "br_vocab_stats")
        off = np.empty(n.value + 1, np.int64)
        pool = np.empty(max(nb.value, 1), np.uint8)
        with torch.cuda.device(self.device):
            check(lib.br_vocab_export(self._h, off.ctypes.data, pool.ctypes.data), "br_vocab_export")
        return off, pool[:nb.value]

    @property
    def terms(self):
        """term id -> str (decoded lazily; the dict-valued attributes of BM25 need it, queries do not)."""
        if self._terms is None:
            off, pool = self._export()
            raw = pool.tobytes()
            o = off.tolist()
            self._terms = [raw[o[i]:o[i + 1]].decode("utf-8") for i in range(len(o) - 1)]
        return self._terms

    # ------------------------------------------------------------------ pickling
    def __getstate__(self):
        off, pool = self._export()
        return dict(pool_off=off, pool=pool, bigrams=self.bigrams)

    def __setstate__(self, st):
        lib = _lib.load()
        dev = _lib.require_cuda(None)
        off = np.ascontiguousarray(st["pool_off"], np.int64)
        pool = np.ascontiguousarray(st["pool"], np.uint8)
        h = C.c_void_p()
        with torch.cuda.device(dev):
            check(lib.br_vocab_import(off.ctypes.data, pool.ctypes.data if pool.size else None, off.size - 1,
                                      _lib.stream_ptr(dev), C.byref(h)), "br_vocab_import")
        self.__init__(h, dev, st["bigrams"])

    @classmethod
    def from_terms(cls, terms, bigrams=False, device=None):
        """Vocabulary with term id = position in ``terms`` (distinct strings)."""
        terms = [str(t) for t in terms]
        if len(set(terms)) != len(terms):
            raise _lib.VocabularyNotDistinct("vocabulary terms are not distinct as strings")
        data, off = pack_texts(terms)
        self = cls.__new__(cls)
        self.__setstate__(dict(pool_off=off, pool=data, bigrams=bigrams))
        return self

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().br_vocab_destroy(self._h)
                self._h = None
        except Exception:
            pass
