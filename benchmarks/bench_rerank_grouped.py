"""Config 3 at sentence granularity (one process, one GPU) -> profiles/bench_rerank_grouped.json.

Workload: the config-3 corpus (C2 'en', 207,363 documents, BM25 built as in bench_c3.py), 10 k queries.  Every document
gets 1 + floor(31 u^3) sentence rows (the distribution of bench_cosine_grouped.py): ~1.8 M x 768 bf16 rows, ~2.8 GB, more
than the 126 MB L2 holds, so the gather reads HBM.  Stages, CUDA events, best of --reps after one warm-up call:
  bm25_top1000            BM25 top-1000 documents per query
  rerank_groups_k10/_k100 CosineIndex.rerank_groups over those documents' rows
  rows_rerank_k10         for comparison on the same rows: CosineIndex.rerank over every query's expanded rows, padded with
                          -1 to the longest expansion
Then one torch.profiler pass per re-rank (separate from the timed runs) for the gather kernels' own device time.  Rates
are gathered bytes (sum over queries of rows x d x 2) over time, also as a fraction of the HBM traffic rate (read +
write) of a plain 4 GiB device-to-device tensor copy timed in the same run.  The card's name and power limit are read
(never set) in the same run."""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench_cosine_grouped import card, kernel_times  # noqa: E402


def best_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return min(out)


def expand_rows(cand, off, sizes):
    """Candidate documents [Q, c] -> every query's sentence rows [Q, R_max] (int32, -1 padded), in candidate order."""
    Q = cand.shape[0]
    g = cand.to(torch.int64)
    cnt = torch.where(g >= 0, sizes[g.clamp(min=0)], 0).flatten()
    start = torch.where(g >= 0, off[g.clamp(min=0)], 0).flatten()
    per_q = cnt.view(Q, -1).sum(1)
    width = int(per_q.max())
    flat = torch.repeat_interleave(torch.arange(cnt.numel(), device=g.device), cnt)       # candidate slot of each row
    first = torch.cumsum(cnt, 0) - cnt
    row = start[flat] + torch.arange(flat.numel(), device=g.device) - first[flat]
    q = flat // g.shape[1]
    col = torch.arange(flat.numel(), device=g.device) - (torch.cumsum(per_q, 0) - per_q)[q]
    out = torch.full((Q, width), -1, dtype=torch.int32, device=g.device)
    out[q, col] = row.to(torch.int32)
    return out, per_q


def main():
    from document_retrieval_b200 import BM25, synth
    from document_retrieval_b200.cosine import CosineIndex
    p = argparse.ArgumentParser()
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--no-profile", action="store_true")
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_rerank_grouped.json"))
    a = p.parse_args()
    nq, dim = a.queries, 768
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
    off = torch.cumsum(sizes, 0) - sizes
    n_rows = int(sizes.sum())
    emb = torch.empty(n_rows, dim, dtype=torch.bfloat16, device=dev)
    for s in range(0, n_rows, 1 << 18):
        e = min(n_rows, s + (1 << 18))
        emb[s:e] = torch.randn(e - s, dim, generator=g, device=dev).to(torch.bfloat16)
    qe = torch.randn(nq, dim, generator=g, device=dev).to(torch.bfloat16)
    rg = torch.repeat_interleave(torch.arange(n, device=dev), sizes)
    ix = CosineIndex(emb, device=dev, row_group=rg, n_groups=n)
    out["workload"] = (f"C2 en: {n} documents, BM25 top-1000, {n_rows} x {dim} bf16 sentence rows "
                       f"({n_rows * dim * 2 / 1e9:.2f} GB, 1 + floor(31 u^3) per document), {nq} queries")

    cand, _ = m.retrieve_top_n_batch(queries, 1000)
    rows, per_q = expand_rows(cand, off, sizes)
    gathered = int(per_q.sum()) * dim * 2
    out["rows_per_query"] = {"mean": float(per_q.double().mean()), "max": int(per_q.max()), "padded_width": rows.shape[1]}
    out["gathered_bytes"] = gathered

    copy_bytes = 4 << 30
    src = torch.empty(copy_bytes, dtype=torch.uint8, device=dev).fill_(1)
    dst = torch.empty_like(src)
    copy_ms = best_ms(lambda: dst.copy_(src), a.reps)
    del src, dst
    copy_traffic = 2 * copy_bytes / (copy_ms * 1e-3)
    out["d2d_copy"] = {"bytes": copy_bytes, "ms": copy_ms, "hbm_traffic_bytes_per_s": copy_traffic}

    cases = {
        "bm25_top1000": lambda: m.retrieve_top_n_batch(queries, 1000),
        "rerank_groups_k10": lambda: ix.rerank_groups(qe, cand, 10),
        "rerank_groups_k100": lambda: ix.rerank_groups(qe, cand, 100),
        "rows_rerank_k10": lambda: ix.rerank(qe, rows, 10),
    }
    res = {}
    for name, fn in cases.items():
        ms = best_ms(fn, a.reps)
        res[name] = {"ms": ms}
        if name != "bm25_top1000":
            res[name]["gathered_bytes_per_s"] = gathered / (ms * 1e-3)
            res[name]["fraction_of_copy_traffic_rate"] = gathered / (ms * 1e-3) / copy_traffic
        print(name, json.dumps(res[name]), flush=True)
    # the grouped result against the row path's: the best row of each query is in its best document
    gi, _ = ix.rerank_groups(qe, cand, 10)
    ri, _ = ix.rerank(qe, rows, 10)
    res["rerank_groups_k10"]["top1_is_group_of_rows_top1"] = float((gi[:, 0].to(torch.int64) == rg[ri[:, 0].to(torch.int64)]).double().mean())
    out["cases"] = res
    if not a.no_profile:
        kern = {}
        for name, key in (("rerank_groups_k10", "k_cosine_rerank_grouped"), ("rows_rerank_k10", "k_cosine_rerank<")):
            kt = kernel_times(cases[name])
            ms = sum(v["ms"] for k, v in kt.items() if key in k)
            kern[name] = {"gather_kernel_ms": ms, "gathered_bytes_per_s": gathered / (ms * 1e-3),
                          "fraction_of_copy_traffic_rate": gathered / (ms * 1e-3) / copy_traffic, "kernels": kt}
            print(name, "gather kernel", ms, "ms", flush=True)
        out["kernels"] = kern
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "kernels"}))


if __name__ == "__main__":
    main()
