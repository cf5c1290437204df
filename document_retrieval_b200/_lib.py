"""ctypes binding of include/br_b200.h (the C-ABI shared library libbr_b200.so, built in-tree by
build.py).  There is no CPU fallback: importing works anywhere (so that host-side logic is testable),
but every compute entry point needs the CUDA library and a B200, and fails loudly otherwise."""
from __future__ import annotations

import ctypes as C
import os

import torch  # noqa: F401  (initialises the CUDA primary context the library shares)

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("BR_B200_SO") or os.path.join(_HERE, "libbr_b200.so")   # BR_B200_SO: build-variant experiments

VARIANT_ID = {"notebook": 0, "okapi": 1, "okapi_no_plus1": 2}
BR_MAX_K = 1024

# name -> (restype, argtypes); mirrors include/br_b200.h one to one
_P = C.c_void_p
SIGNATURES = {
    "br_last_error": (C.c_char_p, []),
    "br_version": (C.c_char_p, []),
    "br_index_build": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int64, _P, C.POINTER(_P)]),
    "br_index_finalize": (C.c_int, [_P, C.c_double, C.c_double, C.c_int, C.c_double, C.c_double, _P, _P]),
    "br_index_destroy": (None, [_P]),
    "br_index_append": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P]),
    "br_index_remove": (C.c_int, [_P, _P, _P]),
    "br_index_stats": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                                 C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "br_index_stats_in_force": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "br_index_df_dev": (_P, [_P]),
    "br_index_export_df_idf": (C.c_int, [_P, _P, _P]),
    "br_index_export_csr": (C.c_int, [_P, _P, _P, _P, _P]),
    "br_index_import_csr": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int64, _P, C.POINTER(_P)]),
    "br_index_export_csr_dev": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "br_index_import_csr_dev": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _P, C.POINTER(_P)]),
    "br_score_batch": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int, _P, _P]),
    "br_topk_batch": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, _P, _P, _P, _P]),
    "br_topk_batch_records": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, _P, _P, _P]),
    "br_topk_batch_filtered": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, _P, _P, _P, _P, _P]),
    "br_topk_batch_records_filtered": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, _P, _P, _P,
                                                 _P]),
    "br_topk_merge_records": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P]),
    "br_rescore_docs": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int, _P, _P, _P, _P]),
    "br_index_enable_tfidf": (C.c_int, [_P, _P]),
    "br_tfidf_cosine_topk": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "br_rerank_v3_scores": (C.c_int, [_P, _P, _P, C.c_int32, _P, _P, _P, _P]),
    "br_topk_merge": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P]),
    "br_row_inv_norms": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P]),
    "br_cosine_topk": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P]),
    "br_cosine_topk_filtered": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P,
                                          _P]),
    "br_cosine_topk_grouped": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int64,
                                         _P, _P, _P, _P]),
    "br_set_cosine_option": (C.c_int, [C.c_char_p, C.c_int]),
    "br_cosine_rerank": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, C.c_int32, _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "br_cosine_rerank_grouped": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, C.c_int32, _P, C.c_int32, _P, C.c_int32, C.c_int32,
                                           _P, _P, _P]),
    "br_fuse_rrf": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int64, C.c_int32, C.c_double, C.c_double, C.c_double,
                              C.c_int32, _P, _P, _P, _P]),
    "br_fuse_linear": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int, _P, _P, C.c_int64, C.c_int32, _P, _P, _P,
                                 C.c_int32, _P, C.c_int32, C.c_double, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "br_dedupe_first_docs": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "br_set_thr_exchange": (C.c_int, [_P, _P, _P, C.c_int, C.c_int]),
    "br_tile_launch_count": (C.c_int, [_P, C.c_int32]),
    "br_trim_scratch": (C.c_int, []),
    "br_last_query_stats": (C.c_int, [_P, _P]),
    "br_set_profiling": (C.c_int, [_P, C.c_int]),
    "br_set_option": (C.c_int, [_P, C.c_char_p, C.c_int]),
    "br_tokenize_count": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, C.POINTER(C.c_int64), _P]),
    "br_vocab_build": (C.c_int, [_P, _P, C.c_int64, C.c_int, _P, C.c_int64, _P, _P, C.POINTER(_P)]),
    "br_vocab_lookup": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, _P, C.c_int64, _P, _P]),
    "br_vocab_extend": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int, _P, C.c_int64, _P, _P]),
    "br_vocab_stats": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "br_vocab_export": (C.c_int, [_P, _P, _P]),
    "br_vocab_import": (C.c_int, [_P, _P, C.c_int64, _P, C.POINTER(_P)]),
    "br_vocab_destroy": (None, [_P]),
}


THR_EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p)


class QueryStats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("queries_fused", C.c_int64), ("queries_dense", C.c_int64),
                ("candidates_rescored", C.c_int64), ("postings_bytes", C.c_int64), ("score_launches", C.c_int64),
                ("score_ms", C.c_double)]


class DocFilterC(C.Structure):
    """br_doc_filter (include/br_b200.h)."""
    _fields_ = [("bits_dev", C.c_void_p), ("words", C.c_int64), ("n_rows", C.c_int32), ("query_row_dev", C.c_void_p)]


class BRError(RuntimeError):
    pass


def _bit_weights(dev):
    return torch.bitwise_left_shift(torch.ones(32, dtype=torch.int64, device=dev), torch.arange(32, device=dev))


def pack_doc_filter(doc_filter=None, query_filter=None, nq: int = 0, n_docs: int = 0, device=None):
    """``doc_filter`` bool [N] (one allow-list for the whole batch) or [F, N] with ``query_filter`` int [Q] (the row each
    query uses, -1 = unfiltered) -> (br_doc_filter struct, tensors it points to); (None, None) without a filter, which
    the library takes as the unfiltered call.  The bits are packed on the device: bit (d & 31) of word (d >> 5) of row
    f = doc_filter[f, d].  Shape mismatches raise ValueError; a query_filter value outside [-1, F) is left to the
    library, which rejects it (BRError)."""
    if doc_filter is None:
        if query_filter is not None:
            raise ValueError("query_filter needs a doc_filter")
        return None, None
    f = torch.as_tensor(doc_filter)
    if f.dtype != torch.bool:
        raise ValueError(f"doc_filter must be a bool array, got {f.dtype}")
    if f.dim() not in (1, 2) or f.shape[-1] != n_docs:
        raise ValueError(f"doc_filter must have shape [{n_docs}] or [F, {n_docs}], got {tuple(f.shape)}")
    if f.dim() == 1:
        if query_filter is not None:
            raise ValueError("query_filter needs a 2-D doc_filter [F, N]")
        f = f[None]
    elif query_filter is None:
        raise ValueError("a 2-D doc_filter [F, N] needs query_filter (int [Q], the row of each query, -1 = unfiltered)")
    n_rows = f.shape[0]
    if n_rows < 1:
        raise ValueError("doc_filter has no rows")
    f = f.to(device).contiguous()
    words = max(1, (n_docs + 31) // 32)
    pad = words * 32 - n_docs
    if pad:
        f = torch.nn.functional.pad(f, (0, pad))
    packed = (f.view(n_rows, words, 32).to(torch.int64) * _bit_weights(f.device)).sum(-1)
    bits = torch.where(packed >= 2 ** 31, packed - 2 ** 32, packed).to(torch.int32).contiguous()
    rows = None
    if query_filter is not None:
        rows = torch.as_tensor(query_filter)
        if rows.dim() != 1 or rows.shape[0] != nq:
            raise ValueError(f"query_filter must have shape [{nq}], got {tuple(rows.shape)}")
        if rows.dtype.is_floating_point or rows.dtype == torch.bool:
            raise ValueError(f"query_filter must be an integer array, got {rows.dtype}")
        rows = rows.to(device=device, dtype=torch.int32).contiguous()
    st = DocFilterC(bits.data_ptr(), words, n_rows, 0 if rows is None else rows.data_ptr())
    return st, (bits, rows)


class VocabularyNotDistinct(BRError):
    """Vocabulary.from_terms: two terms have the same string form (e.g. the int 1 and the str "1")."""


_lib = None


def load():
    """Load libbr_b200.so (no compute happens here)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(SO_PATH):
            raise BRError(f"{SO_PATH} is missing - run `python -m document_retrieval_b200.build` "
                          "(or __graft_entry__.build()); there is no CPU fallback")
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(status: int, what: str = ""):
    if status != 0:
        msg = load().br_last_error().decode("utf-8", "replace")
        raise BRError(f"{what or 'br_b200'} failed ({status}): {msg}")


def require_cuda(device=None):
    if not torch.cuda.is_available():
        raise BRError("document_retrieval_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise BRError(f"device must be a CUDA device, got {dev}")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()
