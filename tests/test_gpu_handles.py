"""Destroying a library handle returns all of its device memory: an index that has served a filtered batch (its filter
workspace included), a string vocabulary, and an index import that the library rejects part way through."""
import ctypes as C
import gc

import numpy as np
import pytest
import torch

from document_retrieval_b200 import BM25, _lib, synth
from document_retrieval_b200.ingest import Vocabulary

pytestmark = pytest.mark.gpu

BR_ERR_INVALID = -1
CYCLES = 16          # handles created and destroyed per window
WINDOWS = 3          # another process on the card moves its free memory: one window of three has to hold
SLACK = 4 << 20      # bytes; a handle that keeps its filter workspace (~1.3 MB at nq = 2^17) drifts by 20+ MiB
NQ = 1 << 17


def _free_bytes():
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    _lib.check(_lib.load().br_trim_scratch(), "br_trim_scratch")
    return torch.cuda.mem_get_info()[0]


def _assert_cycles_return_memory(cycle):
    cycle()                                   # loads the kernels and creates the library's scratch pool
    drift = []
    for _ in range(WINDOWS):
        before = _free_bytes()
        for _ in range(CYCLES):
            cycle()
        drift.append(before - _free_bytes())
        if drift[-1] <= SLACK:
            return
    pytest.fail(f"device memory in use grew by {[d / 2 ** 20 for d in drift]} MiB over {CYCLES} create/destroy cycles")


@pytest.fixture(scope="module")
def corpus():
    do, tk = synth.make_corpus(20_000, 5_000, 40, (91,))
    return do, tk, 5_000


def test_filtered_index_frees_its_workspaces(corpus):
    do, tk, vocab = corpus
    rng = np.random.Generator(np.random.PCG64(92))
    q_off = np.zeros(NQ + 1, np.int64)
    np.cumsum(rng.integers(1, 3, NQ), out=q_off[1:])               # one- and two-term queries
    q_terms = torch.as_tensor(rng.integers(0, vocab, int(q_off[-1])).astype(np.int32), device="cuda")
    q_off = torch.as_tensor(q_off, device="cuda")
    allowed = torch.as_tensor(rng.random(do.size - 1) < 0.5, device="cuda")

    def cycle():
        m = BM25.from_token_ids(do, tk, vocab, device="cuda:0")
        ids, _ = m.retrieve_top_n_batch((q_terms, q_off), 10, doc_filter=allowed)
        assert ids.shape == (NQ, 10)
        del m, ids

    _assert_cycles_return_memory(cycle)


def test_vocabulary_frees_its_tables():
    # ~108k distinct terms: one vocabulary holds ~2.8 MB of device tables, so 16 kept handles would exceed SLACK tenfold
    do, tk = synth.make_corpus(20_000, 200_000, 40, (93,))
    texts = [" ".join(d) for d in synth.to_strings(do, tk)]

    def cycle():
        voc, doc_off, ids = Vocabulary.from_texts(texts, device="cuda:0")
        assert len(voc) > 0 and doc_off.numel() == len(texts) + 1
        del voc, doc_off, ids

    _assert_cycles_return_memory(cycle)


def test_rejected_import_frees_what_it_allocated(corpus):
    do, tk, vocab = corpus
    csr = dict(BM25.from_token_ids(do, tk, vocab, device="cuda:0")._export_csr())
    n_docs = csr["dl"].size
    csr["doc"] = csr["doc"].copy()
    csr["doc"][-1] = n_docs                                          # a doc id outside [0, n_docs): found on the device
    lib = _lib.load()

    def cycle():
        h = C.c_void_p()
        status = lib.br_index_import_csr(csr["row_ptr"].ctypes.data, csr["doc"].ctypes.data, csr["tf"].ctypes.data,
                                         csr["dl"].ctypes.data, n_docs, vocab, 0, _lib.stream_ptr(torch.device("cuda:0")),
                                         C.byref(h))
        assert status == BR_ERR_INVALID and not h.value

    _assert_cycles_return_memory(cycle)
