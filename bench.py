#!/usr/bin/env python
"""bench.py - BM25 top-10 queries/s on the MS-MARCO-passage-shaped synthetic corpus
(BASELINE.json configs[3]: 8.8M docs x ~60 tokens, 1M-term Zipf vocab, 10k queries), doc-sharded
over --gpus N GPUs of one box with an NCCL all-gather + merge of the per-GPU top-k.

A "step" is one pass of the hot path (score + select + float64 re-score + all-gather + merge) over
the whole 10k-query batch.  Prints ONE JSON line (contract in the task statement):
  value      queries/s with the queries already resident in HBM
  e2e        the same through the public API (BM25 / ShardedBM25.retrieve_top_n_batch) from pinned
             HOST query buffers, H2D + D2H inside the timed region
  roofline   scoring kernel: algorithmic bytes (8 B x sum df of the distinct query terms, SURVEY 8d)
             / its CUDA-event time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the plain-C oracle port (oracle/bm25_oracle.c, query-parallel like the reference's
             process_map) on this box's host cores, on a bounded query sample at full N
`--impl reference` times that CPU port alone (the reference itself is Python and has no
compilable sources; oracle/_ref holds only the port).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_BLOCKS = 8   # the corpus is generated in 8 fixed blocks so that it is identical for 1/2/4/8 GPUs


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--docs", type=int, default=8_800_000)
    p.add_argument("--vocab", type=int, default=1_000_000)
    p.add_argument("--mean-len", type=int, default=60)
    p.add_argument("--queries", type=int, default=10_000)
    p.add_argument("--k", type=int, default=10)
    p.add_argument("--cpu-sample", type=int, default=0, help="queries in the CPU baseline sample (0 = auto)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-secondary", action="store_true", help="skip the cosine / index-file figures of `secondary`")
    p.add_argument("--share-thresholds", type=int, default=-1,
                   help="cross-shard threshold exchange of the doc-sharded index (N > 1): 1 on, 0 off, -1 the library default")
    p.add_argument("--opt", action="append", default=[], metavar="NAME=INT",
                   help="br_set_option on the index (tuning experiments, e.g. defer_pm=800); not used by the driver")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write the ids and scores the last timed step returned as DIR/ids.npy and "
                        "DIR/scores.npy (float64), so that two builds can be compared output for output")
    return p.parse_args()


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ids_checksum(ids_cpu):
    """64-bit BLAKE2b of the [Q, k] int64 id matrix (identical across GPU counts by construction of the corpus)."""
    import hashlib
    return hashlib.blake2b(np.ascontiguousarray(ids_cpu.numpy().astype(np.int64)).tobytes(), digest_size=8).hexdigest()


def limiter_profile():
    """ncu figures of the tile kernel (profiles/r2_tile_limiter.json, written by benchmarks/ncu_limiter.py from an
    `ncu --set full` capture) - attached only with a flag saying whether the profiled source is the shipped one."""
    import hashlib
    path = os.path.join(ROOT, "profiles", "r2_tile_limiter.json")
    if not os.path.isfile(path):
        return None
    with open(path) as f:
        d = json.load(f)
    src = os.path.join(ROOT, d.get("source", ""))
    sha = hashlib.sha256(open(src, "rb").read()).hexdigest() if os.path.isfile(src) else None
    d["profile_matches_shipped_source"] = bool(sha and sha == d.get("source_sha256"))
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        """Samples taken from now on count (the sampler is started before the warm-up so that spawning nvidia-smi and
        its NVML initialisation do not fall into the timed region)."""
        self.first = len(self.rows)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        rows = self.rows[getattr(self, "first", 0):] or self.rows[-1:]
        sm = [float(r[0]) for r in rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def block_bounds(n_docs):
    per = -(-n_docs // N_BLOCKS)
    return [(min(n_docs, b * per), min(n_docs, (b + 1) * per)) for b in range(N_BLOCKS)]


def gen_blocks(args, blocks, device):
    """Token ids of the given corpus blocks, generated on the device (synth-v1 distribution)."""
    import torch
    from document_retrieval_b200 import synth
    offs, toks = [], []
    base = 0
    for b in blocks:
        lo, hi = block_bounds(args.docs)[b]
        if hi <= lo:
            continue
        do, tk = synth.make_corpus_torch(hi - lo, args.vocab, args.mean_len, device, seed=synth.ROOT_SEED + 17 * b)
        offs.append(do[:-1] + base if offs else do[:-1])
        base += int(do[-1].item())
        toks.append(tk)
    doc_offsets = torch.cat(offs + [torch.tensor([base], dtype=torch.int64, device=device)])
    return doc_offsets, torch.cat(toks)


def gen_queries(args, doc_offsets, token_ids, doc_lo, doc_hi, rank, world):
    """Queries whose source doc falls in [doc_lo, doc_hi) are built by the owning rank, then gathered."""
    import torch
    import torch.distributed as dist
    rng = np.random.Generator(np.random.PCG64(20241105 + 4))
    src = rng.integers(0, args.docs, size=args.queries)
    m = rng.integers(5, 16, size=args.queries)
    mine = np.nonzero((src >= doc_lo) & (src < doc_hi))[0]
    local = {}
    if mine.size:
        s = torch.from_numpy(src[mine] - doc_lo).to(doc_offsets.device)
        lo = doc_offsets[s].cpu().numpy()
        hi = doc_offsets[s + 1].cpu().numpy()
        width = int((hi - lo).max())
        idx = torch.from_numpy(lo).to(doc_offsets.device)[:, None] + torch.arange(width, device=doc_offsets.device)[None, :]
        toks = token_ids[idx.clamp_(max=token_ids.numel() - 1)].cpu().numpy()
        for j, qi in enumerate(mine.tolist()):
            ln = int(hi[j] - lo[j])
            take = min(int(m[qi]), ln)
            pos = np.random.Generator(np.random.PCG64(977 * qi + 13)).choice(ln, size=take, replace=False)
            t = toks[j, pos].astype(np.int32)
            if qi % 100 == 99:
                t = np.concatenate([t, np.array([args.vocab], np.int32)])     # OOV token
            local[qi] = t
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, local)
        for g in gathered:
            local.update(g)
    terms = [local[i] for i in range(args.queries)]
    q_off = np.zeros(args.queries + 1, np.int32)
    np.cumsum([t.size for t in terms], out=q_off[1:])
    return np.concatenate(terms).astype(np.int32), q_off, src


def dump_outputs(path, ids, scores):
    """The [Q, k] ids and scores of a retrieval call as path/ids.npy and path/scores.npy, both float64 (exact for doc ids
    below 2^53; -1 pads stay -1)."""
    os.makedirs(path, exist_ok=True)
    for name, a in (("ids", ids), ("scores", scores)):
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


def cpu_sample_size(args, threads):
    """Queries in the CPU sample: about 10-15 s of work (one core scores ~9 postings-heavy queries/s at
    N = 8.8M; the cost is linear in N)."""
    per_core_qps = 9.0 * 8_800_000 / max(args.docs, 1)
    return int(max(threads, min(args.queries, per_core_qps * threads * 12)))


def cpu_oracle_run(args, doc_offsets_h, token_ids_h, q_terms, q_off, n_sample, threads, repeats=1):
    """Times the plain-C port on the host: index build (untimed) then `n_sample` queries."""
    from oracle.c_oracle import COracle
    t0 = time.time()
    co = COracle(doc_offsets_h, token_ids_h, args.vocab, variant="notebook", n_threads=threads)
    build_s = time.time() - t0
    qo = q_off[:n_sample + 1]
    best = None
    out = None
    for _ in range(repeats):
        t0 = time.time()
        out = co.topk_batch(q_terms[:qo[-1]], qo, args.k, dedup=True, n_threads=threads)
        dt = time.time() - t0
        best = dt if best is None else min(best, dt)
    return n_sample / best, build_s, best, out



def secondary_benchmarks(args, dev, rank, world, dist_on, model=None, q_dev=None, ids_ref=None):
    """Figures of the other rows of the hot path, measured in the same run so that they are on the driver's record
    (each with its own clock samples): the brute-force cosine GEMM (BASELINE config 5: 1.25 M x 768 bf16 rows per GPU,
    10k queries - the whole 10 M-row config when run on 8 GPUs), the candidate re-rank (config 3) and the index file."""
    import torch
    import torch.distributed as dist
    from document_retrieval_b200.cosine import CosineIndex
    from document_retrieval_b200.sharded import ShardedCosineIndex
    out = {}
    peaks = {}
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            peaks = json.load(f)
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    tf_burst = float(peaks.get("bf16_tflops", 1590.0))
    tf_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    steps, warm = max(3, min(args.steps, 10)), 3

    def timed(fn):
        for _ in range(warm):
            fn()
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            r = fn()
        e1.record()
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if dist_on:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, r

    # ---- config 5: brute-force cosine top-10, 1.25 M rows per GPU
    n_rows, dim, nq = 1_250_000, 768, args.queries
    g = torch.Generator(device=dev).manual_seed(20241105 + 5 + 1000 * rank)
    docs = torch.empty(n_rows, dim, device=dev, dtype=torch.bfloat16)
    for a in range(0, n_rows, 1 << 18):
        b = min(n_rows, a + (1 << 18))
        docs[a:b] = torch.randn(b - a, dim, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)
    gq = torch.Generator(device=dev).manual_seed(20241105 + 55)
    qs = torch.randn(nq, dim, generator=gq, device=dev, dtype=torch.float32).to(torch.bfloat16)
    ix = ShardedCosineIndex(docs, rank * n_rows, device=dev)
    sampler = ClockSampler(dev.index or 0)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
        sampler.mark()
    ms, (ids, sims) = timed(lambda: ix.topk(qs, 10))
    clocks = sampler.stop() if rank == 0 else None
    # ids against torch fp32 on a 256-query sample of this rank's rows (canonical side: torch.topk on fp32 of the bf16
    # values, team_run1.py:270-282; near-ties within 2e-6 may order differently - counted separately)
    ns = 256
    li, ls = ix.local.topk(qs[:ns], 10)
    same = near = 0
    qn = qs[:ns].float()
    qn = qn / (qn.norm(dim=1, keepdim=True) + 1e-10)
    best = torch.full((ns, 10), -2.0, device=dev)
    best_i = torch.zeros((ns, 10), dtype=torch.int64, device=dev)
    for a in range(0, n_rows, 1 << 18):
        b = min(n_rows, a + (1 << 18))
        dn = docs[a:b].float()
        dn = dn / (dn.norm(dim=1, keepdim=True) + 1e-10)
        sc = qn @ dn.T
        v, i = torch.topk(torch.cat([best, sc], 1), 10, dim=1)
        cat_i = torch.cat([best_i, torch.arange(a, b, device=dev).expand(ns, -1)], 1)
        best, best_i = v, torch.gather(cat_i, 1, i)
    li_local = li - rank * n_rows
    eq = (li_local == best_i)
    same = float(eq.all(dim=1).float().mean().item())
    near = float(((ls - best).abs().max(dim=1).values < 2e-6).float().mean().item())
    flop = 2.0 * n_rows * world * nq * dim
    tfs = flop / (ms * 1e-3) / 1e12 / world
    out["cosine_c5"] = {
        "workload": f"BASELINE config 5: {n_rows * world} x {dim} bf16 rows over {world} GPU(s) ({n_rows} per GPU), {nq} queries, "
                    "exact top-10; whole call (tcgen05 GEMM launches + tighten kernels + norms" + (" + NCCL all-gather + merge)" if dist_on else ")"),
        "ms": ms, "queries_per_s": nq / (ms * 1e-3), "tflops_per_gpu": tfs, "frac_of_bf16_burst": tfs / tf_burst,
        "frac_of_bf16_sustained": tfs / tf_sus, "clocks": clocks,
        "check": {"sample_queries": ns, "top10_ids_identical_to_torch_fp32_frac": same,
                  "top10_sims_within_2e-6_frac": near}}
    del ix, docs
    torch.cuda.empty_cache()

    # ---- config 3: BM25 top-1000 -> cosine re-rank, C2 'en'-shaped corpus (rank 0; the other ranks wait)
    if rank == 0:
        from document_retrieval_b200 import BM25, synth
        n3, v3 = 207_363, 200_000
        do3, tk3 = synth.make_corpus_torch(n3, v3, 200, dev, seed=synth.ROOT_SEED + 33)
        qo3, qt3, _ = synth.make_queries_torch(do3, tk3, nq, v3, seed=synth.ROOT_SEED + 34)
        m3 = BM25.from_token_ids(do3, tk3, v3, device=dev)
        del do3, tk3
        emb = torch.randn(n3, dim, generator=gq, device=dev, dtype=torch.float32).to(torch.bfloat16)
        ci = CosineIndex(emb)
        q3 = (torch.from_numpy(qt3).to(dev), torch.from_numpy(qo3).to(dev))
        sampler = ClockSampler(dev.index or 0)
        sampler.start()
        time.sleep(0.3)
        sampler.mark()
        dist_saved, dist_on3 = dist_on, False

        def t3(fn):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                r = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / steps, r
        ms_b, (cand, _) = t3(lambda: m3.retrieve_top_n_batch(q3, 1000))
        ms_r, (ri, rs) = t3(lambda: ci.rerank(qs, cand, 10))
        clocks3 = sampler.stop()
        bytes3 = nq * (1000 * dim * 2 + dim * 2 + 80)
        out["rerank_c3"] = {
            "workload": f"BASELINE config 3: {n3} docs x ~200 tok ({v3}-term vocab), {nq} queries: BM25 top-1000 (fused tiled path, "
                        f"k > 32) then cosine re-rank of the 1000 candidates ({dim}-d bf16) to top-10",
            "bm25_top1000_ms": ms_b, "rerank_ms": ms_r, "queries_per_s": nq / ((ms_b + ms_r) * 1e-3),
            "rerank_GB/s": bytes3 / (ms_r * 1e-3) / 1e9, "rerank_frac_of_hbm": bytes3 / (ms_r * 1e-3) / 1e9 / hbm,
            "note": "re-rank algorithmic bytes = c*D*2 + D*2 + 8k per query (SURVEY 8d); gather-bound", "clocks": clocks3}
        del m3, ci, emb
        torch.cuda.empty_cache()
    # ---- configs 1 and 2 (small corpora: the reference's own CPU-runnable cases), ids checked against the C oracle
    if rank == 0 and world == 1:
        from document_retrieval_b200 import BM25, synth
        from oracle.c_oracle import COracle
        threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

        def t_small(fn, reps=20):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                r = fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps, r
        c1 = synth.make_config("C1")
        t0 = time.time()
        m1 = BM25.from_token_ids(c1["doc_offsets"], c1["token_ids"], c1["vocab"], device=dev)
        torch.cuda.synchronize()
        b1 = time.time() - t0
        q1 = (torch.from_numpy(c1["q_terms"]).to(dev), torch.from_numpy(c1["q_offsets"]).to(dev))
        ms1, (i1, s1) = t_small(lambda: m1.retrieve_top_n_batch(q1, 10))
        co = COracle(c1["doc_offsets"], c1["token_ids"], c1["vocab"], n_threads=threads)
        t0 = time.time()
        oi, osc, _ = co.topk_batch(c1["q_terms"], c1["q_offsets"], 10, n_threads=threads)
        cpu1 = time.time() - t0
        nq1 = c1["q_offsets"].size - 1
        out["bm25_c1"] = {"workload": f"BASELINE config 1: {c1['n_docs']} docs x ~200 tok, {c1['vocab']}-term vocab, {nq1} queries, top-10",
                          "ms_per_batch": ms1, "queries_per_s": nq1 / (ms1 * 1e-3), "index_build_s": b1,
                          "ids_and_float64_scores_identical_to_oracle": bool(np.array_equal(i1.cpu().numpy(), oi) and np.array_equal(s1.cpu().numpy(), osc)),
                          "cpu_port_queries_per_s": nq1 / cpu1, "cpu_cores": threads}
        del m1, co
        langs, queries = synth.make_c2(scale=1.0)
        models, oracles = {}, {}
        t0 = time.time()
        for lang, c in langs.items():
            models[lang] = BM25.from_token_ids(c["doc_offsets"], c["token_ids"], c["vocab"], device=dev)
        torch.cuda.synchronize()
        b2 = time.time() - t0
        by_lang = {}
        for i, q in enumerate(queries):
            by_lang.setdefault(q["lang"], []).append(i)
        packed = {}
        for lang, idxs in by_lang.items():
            terms = np.concatenate([queries[i]["terms"] for i in idxs]).astype(np.int32)
            offs = np.cumsum([0] + [queries[i]["terms"].size for i in idxs]).astype(np.int32)
            packed[lang] = (torch.from_numpy(terms).to(dev), torch.from_numpy(offs).to(dev), terms, offs)

        def run_c2():
            return {lang: models[lang].retrieve_top_n_batch((p[0], p[1]), 10)[0] for lang, p in packed.items()}
        ms2, res2 = t_small(run_c2, reps=10)
        same, hits, cpu2 = True, 0, 0.0
        for lang, idxs in by_lang.items():
            c = langs[lang]
            co = COracle(c["doc_offsets"], c["token_ids"], c["vocab"], n_threads=threads)
            t0 = time.time()
            oi, _, _ = co.topk_batch(packed[lang][2], packed[lang][3], 10, n_threads=threads)
            cpu2 += time.time() - t0
            got = res2[lang].cpu().numpy()
            same = same and bool(np.array_equal(got, oi))
            hits += sum(1 for j, i in enumerate(idxs) if queries[i]["qrel"] in got[j].tolist())
            del co
        out["bm25_c2"] = {"workload": f"BASELINE config 2: 7 per-language indexes, {sum(c['n_docs'] for c in langs.values())} docs, "
                                      f"{len(queries)} mixed-language queries routed by language, top-10",
                          "ms_per_batch": ms2, "queries_per_s": len(queries) / (ms2 * 1e-3), "index_build_s": b2,
                          "recall_at_10": hits / len(queries), "ids_identical_to_oracle": same,
                          "cpu_port_queries_per_s": len(queries) / cpu2, "cpu_cores": threads}
        # TF-IDF cosine candidate stage (cosine_similarity_bm25_reranking.py:210-229) on the largest language index:
        # tiled scorer over the tf*idf^2/||d|| table against the dense scatter-add path it replaced
        big = max(langs, key=lambda l: langs[l]["n_docs"])
        cb = langs[big]
        mt = BM25.from_token_ids(cb["doc_offsets"], cb["token_ids"], cb["vocab"], variant="okapi_no_plus1", dedup_query=False,
                                 device=dev)
        qt = (packed[big][0], packed[big][1])
        mt.tfidf_cosine_top_n_batch(qt, 200)
        ms_t, (it, st_) = t_small(lambda: mt.tfidf_cosine_top_n_batch(qt, 200), reps=5)
        stats_t = mt.query_stats()
        mt.set_option("fused", 0)
        ms_d, (idn, sdn) = t_small(lambda: mt.tfidf_cosine_top_n_batch(qt, 200), reps=2)
        nqt = int(packed[big][3].size - 1)
        out["tfidf_stage"] = {"workload": f"TF-IDF cosine top-200 candidates, largest language index of config 2 ({cb['n_docs']} docs), "
                                          f"{nqt} queries, float64 re-scored band",
                              "ms_per_batch": ms_t, "queries_per_s": nqt / (ms_t * 1e-3),
                              "queries_on_tiled_path": int(stats_t["queries_fused"]), "queries_on_dense_path": int(stats_t["queries_dense"]),
                              "dense_scatter_add_path_ms": ms_d,
                              "identical_to_dense_path": bool(torch.equal(it, idn) and torch.equal(st_, sdn))}
        del models, mt
        torch.cuda.empty_cache()

    # ---- index file: BM25.save / BM25.load of this run's index (flat binary, no pickle) - the step whose joblib
    # counterpart took the reference longer than its retrieval (bm25_ranking.ipynb:222-251)
    if rank == 0 and world == 1 and model is not None:
        import tempfile
        from document_retrieval_b200 import BM25
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "index.brix")
            torch.cuda.synchronize()
            t0 = time.time()
            model.save(path)
            save_s = time.time() - t0
            nbytes = os.path.getsize(path)
            t0 = time.time()
            m2 = BM25.load(path, device=dev)
            torch.cuda.synchronize()
            load_s = time.time() - t0
            ns = min(256, args.queries)
            d_terms, d_off, q_off_h = q_dev
            i2, _ = m2.retrieve_top_n_batch((d_terms[:int(q_off_h[ns])], d_off[:ns + 1]), args.k)
            same = bool(torch.equal(i2.to(torch.int64).cpu(), ids_ref[:ns]))
            del m2
        out["index_file"] = {"bytes": nbytes, "save_s": save_s, "load_s": load_s, "load_GB/s": nbytes / load_s / 1e9,
                             "loaded_index_top10_identical": same,
                             "note": "load = read (page cache: the file was just written) -> pinned staging -> H2D -> device-side "
                                     "validation -> weights, skip tables, rows rebuilt on the GPU; the reference's joblib.load of "
                                     "its dict-of-dicts model is measured at small scale in BASELINE.md"}
        torch.cuda.empty_cache()
    if dist_on:
        dist.barrier()
    return out

_REAL_STDOUT = None


def _quiet_stdout():
    """Everything that libraries print on fd 1 (e.g. NCCL's "NCCL version ..." banner) goes to stderr, so that
    stdout carries exactly the one JSON line of the contract."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(obj):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(obj) + "\n").encode())


def main():
    _quiet_stdout()
    args = parse()
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference" and rank != 0:
        return 0                                              # rank 0 alone runs the CPU arm
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist_on = world > 1 and args.impl == "ours"
    if dist_on:
        dist.init_process_group("nccl", device_id=dev)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    workload = (f"C4 MS-MARCO-shaped synthetic: {args.docs} docs x ~{args.mean_len} tok, {args.vocab}-term Zipf vocab, "
                f"{args.queries} queries of 5-15 terms, BM25 (notebook variant k1=1.5 b=0.75) top-{args.k}")

    # ------------------------------------------------------------------ reference arm (CPU port)
    if args.impl == "reference":
        doc_offsets, token_ids = gen_blocks(args, range(N_BLOCKS), dev)
        q_terms, q_off, _ = gen_queries(args, doc_offsets, token_ids, 0, args.docs, 0, 1)
        do_h, tk_h = doc_offsets.cpu().numpy(), token_ids.cpu().numpy()
        del doc_offsets, token_ids
        n_sample = args.cpu_sample or cpu_sample_size(args, threads)
        from oracle.c_oracle import COracle
        co = COracle(do_h, tk_h, args.vocab, variant="notebook", n_threads=threads)
        qo = q_off[:n_sample + 1]
        for _ in range(args.warmup):
            co.topk_batch(q_terms[:qo[-1]], qo, args.k, dedup=True, n_threads=threads)
        t0 = time.time()
        for _ in range(args.steps):
            ids, sc, _ = co.topk_batch(q_terms[:qo[-1]], qo, args.k, dedup=True, n_threads=threads)
        dt = (time.time() - t0) / args.steps
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ids, sc)
        qps = n_sample / dt
        sample = f"{n_sample} of {args.queries} queries at full N={args.docs} per step, index resident in host RAM"
        _emit(({
            "impl": "reference", "metric": "BM25 top-10 queries/sec", "value": qps, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload},
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ------------------------------------------------------------------ our arm
    from document_retrieval_b200.sharded import ShardedBM25
    blocks_per_rank = N_BLOCKS // world
    my_blocks = list(range(rank * blocks_per_rank, (rank + 1) * blocks_per_rank))
    bb = block_bounds(args.docs)
    doc_lo, doc_hi = bb[my_blocks[0]][0], bb[my_blocks[-1]][1]
    doc_offsets, token_ids = gen_blocks(args, my_blocks, dev)
    q_terms, q_off, src = gen_queries(args, doc_offsets, token_ids, doc_lo, doc_hi, rank, world)
    # untimed warm-up build of a small slice (module loading, allocator warm-up), then the timed build of the shard
    n_warm = min(20_000, int(doc_offsets.numel()) - 1)
    ShardedBM25.from_local_token_ids(doc_offsets[:n_warm + 1], token_ids[:int(doc_offsets[n_warm])], args.vocab,
                                     doc_base=doc_lo, device=dev)
    torch.cuda.synchronize()
    t0 = time.time()
    sh = ShardedBM25.from_local_token_ids(doc_offsets, token_ids, args.vocab, doc_base=doc_lo, device=dev)
    torch.cuda.synchronize()
    build_s = time.time() - t0
    n_tokens_rank = int(token_ids.numel())
    model = sh.local
    if args.share_thresholds >= 0:
        sh.share_thresholds = bool(args.share_thresholds)
    for o in args.opt:
        name, val = o.split("=")
        model.set_option(name, int(val))
    st = model.stats()
    keep_host = (world == 1 and rank == 0 and not args.no_cpu_baseline)
    do_h = doc_offsets.cpu().numpy() if keep_host else None
    tk_h = token_ids.cpu().numpy() if keep_host else None
    del doc_offsets, token_ids
    torch.cuda.empty_cache()

    # queries: pinned host copies (e2e) and device-resident copies (value)
    h_terms = torch.from_numpy(q_terms).pin_memory()
    h_off = torch.from_numpy(q_off).pin_memory()
    d_terms, d_off = h_terms.to(dev), h_off.to(dev)
    h_out = torch.empty((args.queries, args.k), dtype=torch.int64).pin_memory()

    def step_device():
        return sh.retrieve_top_n_batch((d_terms, d_off), args.k)

    def step_e2e():
        ids, _ = sh.retrieve_top_n_batch((h_terms, h_off), args.k)       # H2D inside
        h_out.copy_(ids, non_blocking=True)                               # D2H of the result
        torch.cuda.current_stream().synchronize()
        return h_out

    def barrier():
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (ms for all `steps` calls, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = None
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if dist_on:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                      # before the warm-up: nvidia-smi start-up stays out of the timed region
    for _ in range(args.warmup):
        step_device()
    ids_ref, sc_ref = step_device()
    model.set_profiling(True)
    step_device()                            # creates the profiling events outside the timed region
    sampler.mark()
    ms_total, (ids_last, sc_last) = timed(step_device, args.steps)
    qstats = model.query_stats()            # last step's counters (identical every step)
    clocks = sampler.stop() if rank == 0 else None
    model.set_profiling(False)
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    ids_e2e = h_out.clone()
    assert torch.equal(ids_e2e, ids_ref.cpu()), "e2e and device-resident results differ"

    # the same once more through the STRING surface of the reference (`preprocessed_query.split()` + vocabulary lookup,
    # bm25_ranking.ipynb:341-347): query texts in host memory -> GPU tokeniser / vocabulary lookup -> scoring
    from document_retrieval_b200.ingest import Vocabulary, pack_texts
    voc = Vocabulary.from_terms([f"t{i}" for i in range(args.vocab)], device=dev)
    q_texts = [" ".join(f"t{t}" for t in q_terms[q_off[i]:q_off[i + 1]]) for i in range(args.queries)]
    text_bytes = int(sum(a.nbytes for a in pack_texts(q_texts)))

    def step_text():
        qt, qo = voc.encode_texts(q_texts)
        ids, _ = sh.retrieve_top_n_batch((qt, qo), args.k)
        h_out.copy_(ids, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return h_out

    step_text()
    ms_text, _ = timed(step_text, args.steps)
    assert torch.equal(h_out, ids_ref.cpu()), "text-surface and device-resident results differ"
    del voc

    ms_step = ms_total / args.steps
    qps = args.queries / (ms_step * 1e-3)
    qps_e2e = args.queries / (ms_e2e / args.steps * 1e-3)
    # roofline of the dominant (scoring) kernel on this rank, max-reduced time / summed bytes over ranks
    alg_bytes = float(qstats["postings_bytes"])
    k_ms = float(qstats["score_ms"])
    if dist_on:
        t = torch.tensor([alg_bytes, k_ms], device=dev, dtype=torch.float64)
        tb = t.clone()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        alg_bytes_rank, k_ms = float(tb[0].item()), float(t[1].item())
    else:
        alg_bytes_rank = alg_bytes
    peak, peak_src = measured_peak()
    lim = limiter_profile() if (world == 1 and args.docs == 8_800_000 and args.queries == 10_000) else None
    traffic = lim["dram_bytes"] if (lim and lim["profile_matches_shipped_source"]) else None
    launches = max(1, int(qstats["score_launches"]))
    achieved = alg_bytes_rank / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None
    recall = float(np.mean([(int(src[i]) in ids_e2e[i].tolist()) for i in range(args.queries)]))

    line = {
        "metric": "BM25 top-10 queries/sec", "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sharding": f"docs over {world} GPU(s), NCCL all-gather of [Q,k] + merge",
                   "l2_policy": "inputs (packed postings, %.2f GB per GPU) larger than L2" % (st["nnz"] * 8 / 1e9),
                   "index_build_s": build_s, "postings_per_gpu": st["nnz"], "recall_at_10_vs_source_doc": recall,
                   "ids_checksum": ids_checksum(ids_e2e),
                   "arithmetic": "fp32 accumulation of precomputed posting weights, float64 re-score of the candidate band "
                                 "(ids bit-exact against the float64 reference)"},
        "e2e": {"value": qps_e2e, "unit": "queries/s", "h2d_bytes_per_step": int(h_terms.numel() * 4 + h_off.numel() * 4),
                "d2h_bytes_per_step": int(h_out.numel() * 8)},
        "e2e_text": {"value": args.queries / (ms_text / args.steps * 1e-3), "unit": "queries/s",
                     "h2d_bytes_per_step": text_bytes, "d2h_bytes_per_step": int(h_out.numel() * 8),
                     "note": "queries as preprocessed strings in host memory: Arrow packing, H2D, str.split() + vocabulary lookup "
                             "on the GPU (Vocabulary.encode_texts), then the same scoring call"},
        "gpu_launches": int(qstats["kernel_launches"]) * args.steps,
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "bm25 scoring (per rank)", "achieved": achieved, "peak": peak,
                     "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                     "peak_source": peak_src, "launches_per_step": launches,
                     "algorithmic_bytes_per_launch": alg_bytes_rank / launches,
                     "kernel_ms_per_launch": k_ms / launches, "kernel_share_of_step": k_ms / ms_step,
                     "path": {"fused": int(qstats["queries_fused"]), "dense": int(qstats["queries_dense"])},
                     "limiter": None if lim is None else {
                         "issue_active_pct": lim["issue_active_pct"], "smem_wavefront_pct": lim["smem_wavefront_pct"],
                         "dram_frac": lim["dram_frac"], "l2_hit_pct": lim["l2_hit_pct"], "warps_active_pct": lim["warps_active_pct"],
                         "stall_cycles_per_issue": lim["stall_cycles_per_issue"], "launch_ms": lim["duration_ms"],
                         "launch_inst_executed": lim["inst_executed"], "source": "profiles/r2_tile_limiter.json (ncu --set full)",
                         "profile_matches_shipped_source": lim["profile_matches_shipped_source"],
                         "frac_of_issue_peak": (lim["issue_active_pct"] or 0) / 100.0,
                         "frac_of_hbm_peak_actually_moved": lim["dram_frac"],
                         "binding": "latency at 36% occupancy (3 CTAs/SM: 64 KB of shared-memory accumulators and 80 registers "
                                    "per thread each): long-scoreboard stalls on posting slices, look-up rows and skip-table "
                                    "entries served by L2; neither HBM nor issue slots are saturated",
                         "profiled_launch": "the 256-tile launch (48 % of the step's tiles); `traffic` and "
                                            "`launch_inst_executed` are that launch's, not the average launch's"},
                     "note": "achieved = ALGORITHMIC bytes (8 B x sum df of every query's distinct terms, no credit for "
                             "cross-query reuse or pruning, SURVEY 8d) / CUDA-event time of the scoring kernel launches. The kernel "
                             "does not touch most of those bytes: exact MaxScore deferral streams only the query's rare terms "
                             "(a few % of the postings) and completes the few candidate docs from look-up rows, so `achieved` "
                             "exceeds the HBM peak; `traffic` is the dram byte count of the profiled launch (ncu), `limiter` "
                             "says what the kernel is actually bound by"},
        "index_build": {"s": build_s, "algorithmic_bytes": 4 * n_tokens_rank + 8 * int(st["nnz"]),
                        "GB/s": (4 * n_tokens_rank + 8 * int(st["nnz"])) / build_s / 1e9,
                        "frac": (4 * n_tokens_rank + 8 * int(st["nnz"])) / build_s / 1e9 / peak,
                        "note": "per rank, wall clock around build + statistics all-reduce + finalize (weights, skip tables, rows); "
                                "algorithmic bytes 4 B x tokens + 8 B x postings (SURVEY 8d)"},
    }
    if dist_on:
        # N > 1: rank 0 rebuilds the whole corpus as ONE index and recomputes a query sample - the sharded ids
        # (all-gather + merge over real NCCL) must be identical to it
        ns = min(512, args.queries)
        ok = None
        if rank == 0:
            do_all, tk_all = gen_blocks(args, range(N_BLOCKS), dev)
            from document_retrieval_b200 import BM25
            single = BM25.from_token_ids(do_all, tk_all, args.vocab, device=dev)
            del do_all, tk_all
            si, _ = single.retrieve_top_n_batch((d_terms[:int(q_off[ns])], d_off[:ns + 1]), args.k)
            ok = bool(torch.equal(si.to(torch.int64).cpu(), ids_e2e[:ns]))
            del single
            torch.cuda.empty_cache()
        dist.barrier()
        line["verify"] = {"sample": f"first {ns} queries recomputed on rank 0 against a single (unsharded) index of all "
                                    f"{args.docs} docs", "ids_identical_to_single_index": ok}
    if not args.no_secondary:
        line["secondary"] = secondary_benchmarks(args, dev, rank, world, dist_on, model, (d_terms, d_off, q_off), ids_e2e)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n_sample = args.cpu_sample or cpu_sample_size(args, threads)
        cpu_qps, cpu_build_s, cpu_s, out = cpu_oracle_run(args, do_h, tk_h, q_terms, q_off, n_sample, threads)
        same = bool(np.array_equal(out[0], ids_e2e[:n_sample].numpy().astype(np.int32)))
        line["cpu_baseline"] = {"value": cpu_qps, "unit": "queries/s", "cores": threads, "kind": "port",
                                "sample": f"first {n_sample} of {args.queries} queries at full N={args.docs} "
                                          f"({cpu_s:.1f} s; host index build {cpu_build_s:.1f} s untimed)",
                                "top10_ids_identical_to_gpu": same}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, ids_last, sc_last)
    if rank == 0:
        _emit(line)
    if dist_on:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
