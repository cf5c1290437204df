"""Appending documents to a built index on the flagship workload (one process, one GPU) -> profiles/bench_append.json.

bench.py's C4 corpus (8.8 M docs, 1 M-term Zipf vocabulary, ~60 tokens a doc, same blocks and seeds).  For each n of new
docs: the index of the first N - n docs is built, the last n are appended with br_index_append, and the grown index is
re-finalised with br_index_finalize; the two calls are timed separately with a host clock around work that ends in a
device synchronise (one warm-up append, then --steps appends, each on a freshly built index of the first N - n docs).
For comparison, a full build and finalise of all N docs.  The merge kernel's device time comes from a separate
torch.profiler pass (one more append); its algorithmic bytes are 10 read + 10 written per posting of the grown index
(8-byte posting + 2-byte tf each way).  Every appended index must return the same top-10 ids for bench.py's 10 k queries
as the index built from scratch (ids checksum).  The card's name and power limit are read (never set) in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))


def sync_ms(fn):
    """-> (ms of fn() up to a device synchronise, its result)"""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def merge_kernel_ms(fn):
    """Device time of k_append_merge during fn(), from torch.profiler's CUDA activities."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = [e.device_time_total for e in prof.key_averages() if "k_append_merge" in e.key]
    return sum(us) / 1e3 if us else None


def main():
    import bench
    from bench_filter import card
    from document_retrieval_b200 import BM25, _lib
    from document_retrieval_b200._lib import VARIANT_ID, check, ptr
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--docs", type=int, default=8_800_000)
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--new", type=int, nargs="+", default=[10_000, 100_000, 880_000])
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_append.json"))
    a = p.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    st = _lib.stream_ptr(dev)
    out = {"card": card(), "steps": a.steps, "docs": a.docs, "queries": a.queries, "k": 10}

    args = SimpleNamespace(docs=a.docs, vocab=1_000_000, mean_len=60, queries=a.queries)
    do, tk = bench.gen_blocks(args, range(bench.N_BLOCKS), dev)
    q_terms, q_off, _ = bench.gen_queries(args, do, tk, 0, a.docs, 0, 1)
    q = (torch.from_numpy(q_terms).to(dev), torch.from_numpy(q_off).to(dev))
    N, V = a.docs, args.vocab

    # full build for comparison, and the reference result
    builds, finals = [], []
    ref = None
    for i in range(a.steps + 1):                       # the first build and finalise are the warm-up
        ref = None
        torch.cuda.empty_cache()
        t_b, ref = sync_ms(lambda: BM25.from_token_ids(do, tk, V, device=dev, finalize=False))
        t_f, _ = sync_ms(ref.finalize)
        if i:
            builds.append(t_b)
            finals.append(t_f)
    ids_ref, _ = ref.retrieve_top_n_batch(q, 10)
    out["full"] = {"build_ms": builds, "finalize_ms": finals, "nnz": ref.stats()["nnz"],
                   "ids_checksum": bench.ids_checksum(ids_ref.cpu().to(torch.int64))}
    del ref, ids_ref
    torch.cuda.empty_cache()

    for n in a.new:
        cut = N - n
        do_a, tk_a = do[:cut + 1], tk[:int(do[cut])]
        do_b = (do[cut:] - do[cut]).contiguous()
        tk_b = tk[int(do[cut]):].contiguous()
        v_a = int(tk_a.max()) + 1
        appends, finals = [], []
        m = None
        for i in range(a.steps + 2):
            m = None
            torch.cuda.empty_cache()
            m = BM25.from_token_ids(do_a, tk_a, v_a, device=dev)

            def append():
                check(lib.br_index_append(m._h, ptr(tk_b), ptr(do_b), n, V, st), "br_index_append")

            def finalize():
                check(lib.br_index_finalize(m._h, float(m.k1), float(m.b), VARIANT_ID[m.variant], 0.0, 0.0, None, st),
                      "br_index_finalize")
            if i == a.steps + 1:                       # the profiled pass, kept out of the timed ones
                kernel_ms = merge_kernel_ms(append)
            else:
                t_a, _ = sync_ms(append)
                t_f, _ = sync_ms(finalize)
                if i:                                  # i == 0: warm-up
                    appends.append(t_a)
                    finals.append(t_f)
        finalize()
        m.corpus_size, m.vocab_size = N, V
        m.avgdl = m.stats()["avgdl"]
        ids, _ = m.retrieve_top_n_batch(q, 10)
        nnz = m.stats()["nnz"]
        merge_bytes = 20 * nnz
        out[f"append_{n}"] = {
            "n_new": n, "vocab_before": v_a, "vocab_after": V, "nnz_after": nnz,
            "append_ms": appends, "finalize_ms": finals,
            "merge_kernel_ms": kernel_ms, "merge_bytes": merge_bytes,
            "merge_gbs": None if not kernel_ms else merge_bytes / kernel_ms / 1e6,
            "ids_checksum": bench.ids_checksum(ids.cpu().to(torch.int64))}
        del m, ids
    ok = all(out[f"append_{n}"]["ids_checksum"] == out["full"]["ids_checksum"] for n in a.new)
    out["checksums_equal"] = ok
    print(json.dumps(out, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    assert ok, "an appended index returned other top-10 ids than the index built from scratch"


if __name__ == "__main__":
    main()
