"""CPU simulation (numpy, analysis only): the shape of the tile scorer's essential-posting walk.

Restates make_plan (br_tile.cu) on a reduced synth-v1 corpus: per query, the threshold is set to its true k-th best
score, the streamed-row terms (df >= 0.2 N) are deferred all or nothing, then the other look-up-row terms
(df >= N / 64) smallest bound first while the deferred bounds stay below frac * thr.  What is left and has a skip table
(df >= n_sub / 4) is streamed; rarer terms go through the cold bucket.  Per (query, 2048-doc sub-range) it prints:

  essential postings          postings of the streamed terms in the sub-range
  non-empty essential slices  streamed terms with at least one posting there
  crossing-list entries       docs whose partial score (streamed + cold terms) reaches t1 = thr (1 - 1e-5)^2 - sum ub
  list overflows              sub-ranges with more than 64 crossings (LIST_CAP)
  steps, slice by slice       sum over streamed terms of max(1, ceil(len / 32)): one 32-lane step per slice and chunk
  steps, one stream           ceil(sum len / 32): the slices concatenated

as the mean over all (query, sub-range) pairs and the p50 / p90 over queries of each query's mean.  The thresholds of
a full-size corpus are higher, so more terms are deferred there than here.

    python benchmarks/sim_walk.py [--docs 1100000] [--queries 300]
"""
import argparse
import sys
import time

import numpy as np
import scipy.sparse as sp

sys.path.insert(0, ".")
from document_retrieval_b200 import synth  # noqa: E402

SUB = 2048          # docs per sub-range (kSubShift = 11)
LIST_CAP = 64


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--docs", type=int, default=1_100_000)
    p.add_argument("--vocab", type=int, default=1_000_000)
    p.add_argument("--mean-len", type=int, default=60)
    p.add_argument("--queries", type=int, default=300)
    p.add_argument("--k", type=int, default=10)
    p.add_argument("--frac", type=float, default=0.65, help="deferral budget (defer_pm / 1000)")
    args = p.parse_args()
    t0 = time.time()
    N, V = args.docs, args.vocab
    doc_off, tok = synth.make_corpus(N, V, args.mean_len)
    q_off, q_terms, _ = synth.make_queries(doc_off, tok, args.queries, V)
    dl = np.diff(doc_off)
    doc_of_tok = np.repeat(np.arange(N, dtype=np.int64), dl)
    M = sp.csr_matrix((np.ones(tok.size, np.float32), (tok.astype(np.int64), doc_of_tok)), shape=(V, N))
    M.sum_duplicates()
    M.sort_indices()
    tf = M.data.astype(np.float64)
    df = np.diff(M.indptr)
    term_of = np.repeat(np.arange(V), df)
    idf = np.log(1 + (N - df + 0.5) / (df + 0.5))
    w = idf[term_of] * (tf * 2.5) / (tf + 1.5 * (1 - 0.75 + dl[M.indices] / dl.mean()))
    W = sp.csr_matrix((w.astype(np.float32), M.indices, M.indptr), shape=(V, N))
    ub = np.zeros(V)
    np.maximum.at(ub, term_of, w)
    n_sub = (N + SUB - 1) // SUB
    hot_min = max(4, n_sub // 4)
    row_min, srow_min = N / 64, 0.2 * N

    def per_sub(t):
        return np.bincount(M.indices[M.indptr[t]:M.indptr[t + 1]] // SUB, minlength=n_sub)

    rows = []
    for qi in range(args.queries):
        ts = np.unique(q_terms[q_off[qi]:q_off[qi + 1]])
        ts = ts[(ts >= 0) & (ts < V)]
        ts = ts[df[ts] > 0]
        if ts.size == 0:
            continue
        sc = np.asarray(W[ts].sum(axis=0)).ravel()
        thr = np.partition(sc, -args.k)[-args.k]
        budget = thr * (1 - 1e-5) * args.frac
        look = ts[(df[ts] >= row_min) & (df[ts] >= hot_min)]
        srows = look[df[look] >= srow_min]
        deferred, s = [], 0.0
        if ub[srows].sum() < budget:
            deferred, s = list(srows), ub[srows].sum()
            for t in sorted(set(look) - set(srows), key=lambda t: (ub[t], t)):
                if s + ub[t] >= budget:
                    break
                s += ub[t]
                deferred.append(t)
        ess = [t for t in ts if t not in deferred and df[t] >= hot_min]
        cold = [t for t in ts if df[t] < hot_min]
        lens = np.array([per_sub(t) for t in ess]).reshape(len(ess), n_sub)
        post = lens.sum(axis=0)
        part = ess + cold
        partial = np.asarray(W[np.array(part, np.int64)].sum(axis=0)).ravel() if part else np.zeros(N)
        if deferred:
            t1 = thr * (1 - 1e-5) ** 2 - s
            cross = np.bincount(np.nonzero(partial >= t1)[0] // SUB, minlength=n_sub)
        else:
            cross = np.zeros(n_sub, np.int64)      # no threshold pushes: the sub-range is scanned
        rows.append(np.stack([post, (lens > 0).sum(axis=0), cross, cross > LIST_CAP,
                              np.maximum(1, (lens + 31) // 32).sum(axis=0), (post + 31) // 32]).astype(np.float64))
    names = ["essential postings", "non-empty essential slices", "crossing-list entries (docs >= t1)",
             "sub-ranges with a list overflow", "32-lane walk steps, slice by slice", "32-lane steps of one stream"]
    allv = np.concatenate(rows, axis=1)
    per_q = np.array([r.mean(axis=1) for r in rows])
    print(f"synth-v1, {N} docs, {len(rows)} queries, top-{args.k}, frac {args.frac}; per (query, {SUB}-doc sub-range)")
    print(f"| quantity | mean | p50 query | p90 query |\n|---|---|---|---|")
    for i, n in enumerate(names):
        print(f"| {n} | {allv[i].mean():.1f} | {np.percentile(per_q[:, i], 50):.1f} | {np.percentile(per_q[:, i], 90):.1f} |")
    print(f"({time.time() - t0:.0f} s)")


if __name__ == "__main__":
    main()
