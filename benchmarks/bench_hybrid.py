"""Hybrid retrieval on the config-3 corpus (one process, one GPU) -> profiles/bench_hybrid.json.

Workload: C2 'en', 207,363 documents, BM25 built as in bench_c3.py, 10 k queries, k = 10.  Two dense sides over the same
documents: "flat", one 768-d bf16 embedding per document (0.32 GB), and "grouped", the sentence rows of
bench_rerank_grouped.py (1 + floor(31 u^3) rows per document, ~1.7 M x 768, 2.65 GB).  Both exceed the 126 MB L2, so
the cosine gathers read HBM.  Stages, CUDA events, best of --reps after one warm-up call:
  bm25_top100          BM25 top-100, positive_only (the first stage of hybrid_search)
  dense_top100         CosineIndex.topk (flat) / topk_groups (grouped)
  fuse_rrf             reciprocal rank fusion of the two lists
  fuse_linear          linear fusion: exact BM25 and cosine of the union, min-max normalisation, selection
  hybrid_rrf / _linear whole hybrid_search calls
Then one torch.profiler pass per fusion (separate from the timed runs) for each kernel's own device time.  The
completion's gathered bytes (sum over queries of the union's embedding rows x d x 2) over the cosine gather kernel's
time are set against the HBM traffic rate (read + write) of a 4 GiB device-to-device copy timed in the same run.  The
card's name and power limit are read (never set) in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench_cosine_grouped import card, kernel_times  # noqa: E402
from bench_rerank_grouped import best_ms  # noqa: E402

NEW_KERNELS = ("k_fuse_union", "k_fuse_linear", "k_fuse_components")


def union_rows(B, D, rows_of):
    """-> (union members per query, embedding rows of those members per query); rows_of: rows per document."""
    u = torch.sort(torch.cat([B.to(torch.int64), D.to(torch.int64)], 1), 1).values
    first = torch.ones_like(u, dtype=torch.bool)
    first[:, 1:] = u[:, 1:] != u[:, :-1]
    member = first & (u >= 0)
    return member.sum(1), torch.where(member, rows_of[u.clamp(min=0)], 0).sum(1)


def main():
    from document_retrieval_b200 import BM25, synth
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.hybrid import fuse_linear, fuse_rrf, hybrid_search
    p = argparse.ArgumentParser()
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--no-profile", action="store_true")
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_hybrid.json"))
    a = p.parse_args()
    nq, dim, k, nb, nd = a.queries, 768, 10, 100, 100
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    out = {"card": card(), "reps": a.reps}

    n, vocab = synth.C2_LANG_DOCS["en"], synth.C2_VOCAB["en"]
    do, tk = synth.make_corpus_torch(n, vocab, synth.C2_MEAN_LEN, dev, seed=synth.ROOT_SEED + 2)
    qo, qt, _ = synth.make_queries_torch(do, tk, nq, vocab, seed=synth.ROOT_SEED + 3)
    m = BM25.from_token_ids(do, tk, vocab)
    queries = (torch.from_numpy(qt).to(dev), torch.from_numpy(qo).to(dev))
    g = torch.Generator(device=dev).manual_seed(synth.ROOT_SEED + 3)
    sizes = (1 + torch.floor(31 * torch.rand(n, generator=g, device=dev) ** 3)).to(torch.int64)
    n_rows = int(sizes.sum())

    def rand_rows(r):
        e = torch.empty(r, dim, dtype=torch.bfloat16, device=dev)
        for s in range(0, r, 1 << 18):
            t = min(r, s + (1 << 18))
            e[s:t] = torch.randn(t - s, dim, generator=g, device=dev).to(torch.bfloat16)
        return e

    sides = {
        "flat": (CosineIndex(rand_rows(n), device=dev), torch.ones(n, dtype=torch.int64, device=dev)),
        "grouped": (CosineIndex(rand_rows(n_rows), device=dev, row_group=torch.repeat_interleave(torch.arange(n, device=dev), sizes),
                                n_groups=n), sizes),
    }
    qe = torch.randn(nq, dim, generator=g, device=dev).to(torch.bfloat16)
    out["workload"] = (f"C2 en: {n} documents, {nq} queries, BM25 top-{nb} (positive_only) + dense top-{nd}, k = {k}; "
                       f"flat: {n} x {dim} bf16 (one row per document); grouped: {n_rows} x {dim} bf16 sentence rows "
                       f"({n_rows * dim * 2 / 1e9:.2f} GB, 1 + floor(31 u^3) per document)")

    copy_bytes = 4 << 30
    src = torch.empty(copy_bytes, dtype=torch.uint8, device=dev).fill_(1)
    dst = torch.empty_like(src)
    copy_ms = best_ms(lambda: dst.copy_(src), a.reps)
    del src, dst
    copy_traffic = 2 * copy_bytes / (copy_ms * 1e-3)
    out["d2d_copy"] = {"bytes": copy_bytes, "ms": copy_ms, "hbm_traffic_bytes_per_s": copy_traffic}

    B, _ = m.retrieve_top_n_batch(queries, nb, positive_only=True)
    for side, (ix, rows_of) in sides.items():
        grouped = ix.row_group is not None
        dense = (lambda: ix.topk_groups(qe, nd)) if grouped else (lambda: ix.topk(qe, nd))
        D = dense()[0].to(torch.int32)
        members, rows = union_rows(B, D, rows_of)
        gathered = int(rows.sum()) * dim * 2
        res = {"union_members_per_query": {"mean": float(members.double().mean()), "max": int(members.max())},
               "gathered_bytes": gathered}
        cases = {
            "bm25_top100": lambda: m.retrieve_top_n_batch(queries, nb, positive_only=True),
            "dense_top100": dense,
            "fuse_rrf": lambda: fuse_rrf(B, D, n, k),
            "fuse_linear": lambda: fuse_linear(m, ix, queries, qe, B, D, k),
            "hybrid_rrf": lambda: hybrid_search(m, ix, queries, qe, k, nb, nd, "rrf"),
            "hybrid_linear": lambda: hybrid_search(m, ix, queries, qe, k, nb, nd, "linear"),
        }
        for name, fn in cases.items():
            res[name] = {"ms": best_ms(fn, a.reps)}
            print(side, name, json.dumps(res[name]), flush=True)
        if not a.no_profile:
            gather_key = "k_cosine_rerank_grouped" if grouped else "k_cosine_rerank<"
            for name in ("fuse_rrf", "fuse_linear"):
                kt = kernel_times(cases[name])
                res[name]["kernels"] = kt
                res[name]["new_kernels_ms"] = sum(v["ms"] for key, v in kt.items() if any(s in key for s in NEW_KERNELS))
            kt = res["fuse_linear"]["kernels"]
            g_ms = sum(v["ms"] for key, v in kt.items() if gather_key in key)
            res["fuse_linear"]["completion"] = {
                "gather_kernel_ms": g_ms, "gathered_bytes_per_s": gathered / (g_ms * 1e-3),
                "fraction_of_copy_traffic_rate": gathered / (g_ms * 1e-3) / copy_traffic}
            print(side, "completion", json.dumps(res["fuse_linear"]["completion"]), flush=True)
        out[side] = res
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({s: {c: v["ms"] for c, v in out[s].items() if isinstance(v, dict) and "ms" in v} for s in sides}))


if __name__ == "__main__":
    main()
