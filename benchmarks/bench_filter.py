"""Filtered top-k on the flagship workloads (one process, one GPU) -> profiles/bench_filter.json.

BM25: bench.py's C4 workload (same sizes, blocks and seeds: 8.8 M docs, 1 M-term Zipf vocabulary, 10 k queries, top-10),
retrieved unfiltered, with an all-ones filter, random allow-lists at density 0.5 / 0.1 / 0.01, a contiguous 10 % doc
range and 7 disjoint "language" rows assigned per query.  Per case: queries/s over the timed steps (the filter is packed on
the device inside every call, as a user's call would), tile-kernel ms of the last step (set_profiling /
query_stats().score_ms), queries served by the tiled / dense paths, and an ids checksum.
Cosine: the config-5 shard (1.25 M x 768 bf16 rows, 10 k queries, top-10), unfiltered and at the same densities; whole
call ms.  The card's name and power limit are read (never set) in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, plim, clk = [x.strip() for x in out[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:                     # read-only query; a missing tool is recorded, not fatal
        return {"name": torch.cuda.get_device_name(), "error": repr(e)}


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = None
    for _ in range(steps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps, out


def main():
    import bench
    from document_retrieval_b200 import BM25
    from document_retrieval_b200.cosine import CosineIndex
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--docs", type=int, default=8_800_000)
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--cos-rows", type=int, default=1_250_000)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_filter.json"))
    a = p.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    out = {"card": card(), "steps": a.steps, "warmup": a.warmup}

    # ---- BM25, bench.py's C4 workload
    args = SimpleNamespace(docs=a.docs, vocab=1_000_000, mean_len=60, queries=a.queries)
    do, tk = bench.gen_blocks(args, range(bench.N_BLOCKS), dev)
    q_terms, q_off, _ = bench.gen_queries(args, do, tk, 0, a.docs, 0, 1)
    m = BM25.from_token_ids(do, tk, args.vocab, device=dev)
    del do, tk
    torch.cuda.empty_cache()
    n, nq, k = m.corpus_size, a.queries, 10
    q = (torch.from_numpy(q_terms).to(dev), torch.from_numpy(q_off).to(dev))
    g = torch.Generator(device=dev).manual_seed(20241105 + 99)
    rng_q = torch.Generator(device=dev).manual_seed(20241105 + 98)
    lang = torch.randint(0, 7, (n,), generator=g, device=dev)
    rng_range = torch.zeros(n, dtype=torch.bool, device=dev)
    rng_range[n // 3:n // 3 + n // 10] = True
    cases = {
        "unfiltered": {},
        "all_ones": dict(doc_filter=torch.ones(n, dtype=torch.bool, device=dev)),
        "random_0.5": dict(doc_filter=torch.rand(n, generator=g, device=dev) < 0.5),
        "random_0.1": dict(doc_filter=torch.rand(n, generator=g, device=dev) < 0.1),
        "random_0.01": dict(doc_filter=torch.rand(n, generator=g, device=dev) < 0.01),
        "range_10pct": dict(doc_filter=rng_range),
        "languages_7": dict(doc_filter=torch.stack([lang == i for i in range(7)]),
                            query_filter=torch.randint(0, 7, (nq,), generator=rng_q, device=dev).to(torch.int32)),
    }
    bm = {}
    for name, kw in cases.items():
        ms, (ids, _) = timed(lambda: m.retrieve_top_n_batch(q, k, **kw), a.steps, a.warmup)
        m.set_profiling(True)
        m.retrieve_top_n_batch(q, k, **kw)
        st = m.query_stats()
        m.set_profiling(False)
        bm[name] = {"queries_per_s": nq / (ms * 1e-3), "ms_per_call": ms, "tile_kernel_ms": st["score_ms"],
                    "score_launches": st["score_launches"], "queries_fused": st["queries_fused"],
                    "queries_dense": st["queries_dense"], "ids_checksum": bench.ids_checksum(ids.cpu().to(torch.int64))}
        print(name, json.dumps(bm[name]), flush=True)
    assert bm["all_ones"]["ids_checksum"] == bm["unfiltered"]["ids_checksum"], "an all-ones filter changed the result"
    out["bm25_c4"] = {"workload": f"bench.py C4: {n} docs, 1M-term Zipf vocab, {nq} queries, top-{k}", "cases": bm}
    del m, cases
    torch.cuda.empty_cache()

    # ---- cosine, the config-5 shard
    n_rows, dim = a.cos_rows, 768
    gd = torch.Generator(device=dev).manual_seed(20241105 + 5)
    docs = torch.empty(n_rows, dim, device=dev, dtype=torch.bfloat16)
    for s in range(0, n_rows, 1 << 18):
        e = min(n_rows, s + (1 << 18))
        docs[s:e] = torch.randn(e - s, dim, generator=gd, device=dev, dtype=torch.float32).to(torch.bfloat16)
    qs = torch.randn(nq, dim, generator=torch.Generator(device=dev).manual_seed(20241105 + 55), device=dev,
                     dtype=torch.float32).to(torch.bfloat16)
    ix = CosineIndex(docs, device=dev)
    cos = {}
    for name, dens in (("unfiltered", None), ("random_0.5", 0.5), ("random_0.1", 0.1), ("random_0.01", 0.01)):
        kw = {} if dens is None else dict(doc_filter=torch.rand(n_rows, generator=g, device=dev) < dens)
        ms, (ids, _) = timed(lambda: ix.topk(qs, k, **kw), a.steps, a.warmup)
        cos[name] = {"ms_per_call": ms, "queries_per_s": nq / (ms * 1e-3),
                     "ids_checksum": bench.ids_checksum(ids.cpu().to(torch.int64))}
        print("cosine", name, json.dumps(cos[name]), flush=True)
    out["cosine_c5"] = {"workload": f"config-5 shard: {n_rows} x {dim} bf16 rows, {nq} queries, top-{k}; whole call",
                        "cases": cos}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
