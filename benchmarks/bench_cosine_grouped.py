"""Grouped (document-level) cosine top-k on the config-5 shard (one process, one GPU) -> profiles/bench_cosine_grouped.json.

Workload: 1.25 M x 768 bf16 rows (seeded), grouped into documents of 1-32 sentences (size 1 + floor(31 u^3), mean ~8.75,
~143 k documents); a document's rows are its centre plus Gaussian noise of the same scale (rows of one document have
cosine ~0.5 with each other), 10 k queries are noisy copies of random document centres.  Cases, whole-call ms over the
timed steps:
  topk_k10              ungrouped CosineIndex.topk, k = 10, on the same rows (the baseline)
  groups_k10 / _k100    CosineIndex.topk_groups
  composition           topk(100) + dedupe_sentences_to_docs(10) (team_run1.py:277-294), with the number of queries it
                        leaves with fewer than 10 documents and the agreement of its ids with groups_k10 where it has 10
  groups_k10_filter0.1  topk_groups k = 10 with one random group filter of density 0.1
Then one torch.profiler pass per case (separate from the timed runs): device time per kernel, and launch counts.  The card's
name and power limit are read (never set) in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

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


def kernel_times(fn):
    """One call under torch.profiler -> {kernel name: {"ms": device time, "launches": n}}, largest first."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t > 0:
            out[e.key[:90]] = {"ms": t / 1e3, "launches": e.count}
    return dict(sorted(out.items(), key=lambda kv: -kv[1]["ms"]))


def main():
    import bench
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.sentences import dedupe_sentences_to_docs
    p = argparse.ArgumentParser()
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--rows", type=int, default=1_250_000)
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--no-profile", action="store_true")
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_cosine_grouped.json"))
    a = p.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    out = {"card": card(), "steps": a.steps, "warmup": a.warmup}

    n_rows, dim, nq = a.rows, 768, a.queries
    g = torch.Generator(device=dev).manual_seed(20241105 + 505)
    sizes = []
    total = 0
    while total < n_rows:                                            # documents of 1-32 sentences, mean ~8.75
        s = (1 + torch.floor(31 * torch.rand(65536, generator=g, device=dev) ** 3)).to(torch.int64).cpu()
        sizes.append(s)
        total += int(s.sum())
    sizes = torch.cat(sizes)
    cum = torch.cumsum(sizes, 0)
    n_groups = int(torch.searchsorted(cum, torch.tensor(n_rows)).item()) + 1
    sizes = sizes[:n_groups].clone()
    sizes[-1] -= int(cum[n_groups - 1]) - n_rows
    rg = torch.repeat_interleave(torch.arange(n_groups), sizes).to(dev)
    centres = torch.randn(n_groups, dim, generator=g, device=dev)
    docs = torch.empty(n_rows, dim, device=dev, dtype=torch.bfloat16)
    for s in range(0, n_rows, 1 << 18):
        e = min(n_rows, s + (1 << 18))
        docs[s:e] = (centres[rg[s:e]] + torch.randn(e - s, dim, generator=g, device=dev)).to(torch.bfloat16)
    pick = torch.randint(0, n_groups, (nq,), generator=g, device=dev)
    qs = (centres[pick] + torch.randn(nq, dim, generator=g, device=dev)).to(torch.bfloat16)
    del centres
    gfilter = torch.rand(n_groups, generator=g, device=dev) < 0.1
    rg32 = rg.to(torch.int32)
    ix = CosineIndex(docs, device=dev, row_group=rg, n_groups=n_groups)
    out["workload"] = (f"config-5 shard: {n_rows} x {dim} bf16 rows in {n_groups} documents of 1-32 rows "
                       f"(mean {n_rows / n_groups:.2f}), {nq} queries; whole call")

    def composition():
        rows, _ = ix.topk(qs, 100)
        return dedupe_sentences_to_docs(rows, rg32, 10), None

    cases = {
        "topk_k10": lambda: ix.topk(qs, 10),
        "groups_k10": lambda: ix.topk_groups(qs, 10),
        "groups_k100": lambda: ix.topk_groups(qs, 100),
        "composition": composition,
        "groups_k10_filter0.1": lambda: ix.topk_groups(qs, 10, doc_filter=gfilter),
    }
    res, ids_of = {}, {}
    for name, fn in cases.items():
        ms, (ids, _) = timed(fn, a.steps, a.warmup)
        ids_of[name] = ids
        res[name] = {"ms_per_call": ms, "queries_per_s": nq / (ms * 1e-3),
                     "ids_checksum": bench.ids_checksum(ids.cpu().to(torch.int64))}
        print(name, json.dumps(res[name]), flush=True)
    comp, g10 = ids_of["composition"], ids_of["groups_k10"]
    short = (comp < 0).any(dim=1)
    full = ~short
    res["composition"]["queries_with_fewer_than_10_docs"] = int(short.sum())
    res["composition"]["rows_equal_to_groups_k10_where_10_docs"] = float((comp[full] == g10[full]).all(dim=1).float().mean())
    res["groups_k10"]["valid_ids"] = int((g10 >= 0).sum())
    allowed = gfilter[ids_of["groups_k10_filter0.1"].clamp(min=0)]
    res["groups_k10_filter0.1"]["all_returned_allowed"] = bool(allowed[ids_of["groups_k10_filter0.1"] >= 0].all())
    res["groups_k10"]["ratio_to_topk_k10"] = res["groups_k10"]["ms_per_call"] / res["topk_k10"]["ms_per_call"]
    out["cases"] = res
    if not a.no_profile:
        out["kernels"] = {name: kernel_times(cases[name]) for name in ("topk_k10", "groups_k10", "groups_k100")}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
