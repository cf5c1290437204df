"""Removing documents from a built index on the flagship workload (one process, one GPU) -> profiles/bench_remove.json.

bench.py's C4 corpus (8.8 M docs, 1 M-term Zipf vocabulary, ~60 tokens a doc, same blocks and seeds).  Each case removes a
seeded random set of n docs, or the first n docs as one block (a sliding window), from the index of all N docs with
br_index_remove, then re-finalises it with br_index_finalize; the two calls are timed separately with a host clock around
work that ends in a device synchronise (one warm-up removal, then --steps removals, each from a freshly built index).  For
comparison, a build and finalise of the kept docs from scratch.  The compaction kernels' device time comes from a
separate torch.profiler pass (one more removal).  Their algorithmic bytes are 10 read per posting of the whole index and
10 written per kept posting (8-byte posting + 2-byte tf); the gathers of the doc map, which sit in L2, are not counted.
Every shrunk index must return the same top-10 ids for bench.py's 10 k queries as the index of the kept docs built from
scratch (ids checksum).  The card's name and power limit are read (never set) in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

KERNELS = ("k_remove_count", "k_remove_emit")


def kernel_ms(fn):
    """Device time of each compaction kernel during fn(), from torch.profiler's CUDA activities."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in KERNELS}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                out[k] += e.device_time_total / 1e3
    return out


def main():
    import bench
    from bench_append import sync_ms
    from bench_filter import card
    from document_retrieval_b200 import BM25, _lib
    from document_retrieval_b200._lib import VARIANT_ID, check, ptr
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--docs", type=int, default=8_800_000)
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--remove", type=int, nargs="+", default=[10_000, 100_000, 880_000])
    p.add_argument("--window", type=int, default=880_000, help="also remove the first WINDOW docs as one block")
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_remove.json"))
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
    lens = do[1:] - do[:-1]

    g = torch.Generator(device="cpu").manual_seed(20261022)
    cases = []
    for n in a.remove:
        rm = torch.zeros(N, dtype=torch.bool)
        rm[torch.randperm(N, generator=g)[:n]] = True
        cases.append((f"random_{n}", rm))
    if a.window:
        rm = torch.zeros(N, dtype=torch.bool)
        rm[:a.window] = True
        cases.append((f"first_{a.window}", rm))

    ok = True
    for name, rm in cases:
        rm = rm.to(dev)
        mask = rm.to(torch.uint8)
        keep = ~rm
        n_kept = int(keep.sum())
        do_k = torch.zeros(n_kept + 1, dtype=torch.int64, device=dev)
        torch.cumsum(lens[keep], 0, out=do_k[1:])
        tk_k = tk[torch.repeat_interleave(keep, lens)]

        # the kept docs built from scratch: the reference result, and the time a rebuild takes
        builds, finals = [], []
        for i in range(a.steps + 1):                   # the first build and finalise are the warm-up
            ref = None
            torch.cuda.empty_cache()
            t_b, ref = sync_ms(lambda: BM25.from_token_ids(do_k, tk_k, V, device=dev, finalize=False))
            t_f, _ = sync_ms(ref.finalize)
            if i:
                builds.append(t_b)
                finals.append(t_f)
        ids_ref, _ = ref.retrieve_top_n_batch(q, 10)
        nnz_kept = ref.stats()["nnz"]
        sum_ref = bench.ids_checksum(ids_ref.cpu().to(torch.int64))
        del ref, ids_ref, do_k, tk_k
        torch.cuda.empty_cache()

        removes, finals_r = [], []
        m = None
        kms = None
        for i in range(a.steps + 2):
            m = None
            torch.cuda.empty_cache()
            m = BM25.from_token_ids(do, tk, V, device=dev)
            nnz = m.stats()["nnz"]

            def remove():
                check(lib.br_index_remove(m._h, ptr(mask), st), "br_index_remove")

            def finalize():
                check(lib.br_index_finalize(m._h, float(m.k1), float(m.b), VARIANT_ID[m.variant], 0.0, 0.0, None, st),
                      "br_index_finalize")
            if i == a.steps + 1:                       # the profiled pass, kept out of the timed ones
                kms = kernel_ms(remove)
            else:
                t_r, _ = sync_ms(remove)
                t_f, _ = sync_ms(finalize)
                if i:                                  # i == 0: warm-up
                    removes.append(t_r)
                    finals_r.append(t_f)
        finalize()
        m.corpus_size = n_kept
        m.avgdl = m.stats()["avgdl"]
        ids, _ = m.retrieve_top_n_batch(q, 10)
        assert m.stats()["nnz"] == nnz_kept
        compact_bytes = 10 * nnz + 10 * nnz_kept
        k_ms = sum(kms.values())
        res = {"n_removed": N - n_kept, "n_kept": n_kept, "nnz_before": nnz, "nnz_after": nnz_kept,
               "remove_ms": removes, "finalize_ms": finals_r,
               "rebuild_kept": {"build_ms": builds, "finalize_ms": finals},
               "kernel_ms": kms, "compact_kernels_ms": k_ms, "compact_bytes": compact_bytes,
               "compact_gbs": compact_bytes / k_ms / 1e6 if k_ms else None,
               "ids_checksum": bench.ids_checksum(ids.cpu().to(torch.int64)), "ids_checksum_rebuild": sum_ref}
        res["checksums_equal"] = res["ids_checksum"] == sum_ref
        ok = ok and res["checksums_equal"]
        out[name] = res
        print(name, json.dumps(res), flush=True)
        del m, ids
        torch.cuda.empty_cache()
    out["checksums_equal"] = ok
    print(json.dumps(out, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    assert ok, "a shrunk index returned other top-10 ids than the index of the kept docs built from scratch"


if __name__ == "__main__":
    main()
