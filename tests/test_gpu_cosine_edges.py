"""Dense cosine at the edges of its kernels: ``CosineIndex.topk`` (tcgen05 GEMM + threshold filter, both kernels, with
and without doc filters) and ``CosineIndex.rerank`` / ``br_cosine_rerank`` (the gather kernel that also serves the exact
overflow fallback) against a float64 reference, at dimensions around the 64-wide k-block, the 768 kernel switch and the
16-byte vectors of the gather lanes, corpus sizes around the 128-row CTA half, the 256-row tile and the 64-tile L2
window, query counts around the 112 / 224-query blocks, and on data whose scores are all negative, all near zero, zero,
or exactly tied.

Tolerance from the arithmetic, not tuned: the bf16 inputs and their products are exact; a d-term fp32 sum of them, in
any order, is off by at most (d - 1) 2^-24 sum|q_i x_i|, and the two fp32 norms and three scalings add about
(d + 4) 2^-24 |cos|.  tol = 2 (d + 4) 2^-24 S + 2^-22 with S = sum|q_i x_i| / (||q|| ||x||) covers both, with a
factor 2 for tensor cores that truncate instead of rounding.  The check of the ids is exact given that bound: every
returned row is real, allowed and returned once, the order is (sim desc, id asc), and the returned set can differ from
the reference's only among rows whose reference scores are within 2 tol of the k-th.  The CPU test at the end checks
the bound against torch's own fp32 restatement (oracle.bm25_oracle.cosine_topk)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import bm25_oracle as orc

gpu = pytest.mark.gpu
U = 2.0 ** -24
BIG_BASE = 2 ** 31 + 12345          # ids beyond int32: the int64 id arithmetic of the output


def reference(docs, qs):
    """float64 cosine (q.x) / ((||q|| + 1e-10)(||x|| + 1e-10)) of every (query, row) pair and its tolerance.
    -> (ref float64[Q, N], tol float64[Q, N])"""
    x, q = docs.double(), qs.double()
    nx, nq = x.norm(dim=1), q.norm(dim=1)
    ref = (q @ x.T) / ((nq[:, None] + 1e-10) * (nx[None, :] + 1e-10))
    den = nq[:, None] * nx[None, :]
    s = torch.where(den > 0, (q.abs() @ x.abs().T) / torch.where(den > 0, den, 1.0), 0.0)
    return ref.numpy(), (2 * (docs.shape[1] + 4) * U * s + 2.0 ** -22).numpy()


def check_topk(ids, sims, ref, tol, k, allowed=None, doc_base=0, what=""):
    """Strict check of a top-k answer ids int64[Q, k] (doc_base + row, -1 = padding), sims float32[Q, k] against the
    reference (see the module docstring); ``allowed`` bool[Q, N] or None (every row).  -> largest |sim - ref| / tol."""
    ids, sims = np.asarray(ids, np.int64), np.asarray(sims, np.float32)
    nq, n = ref.shape
    assert ids.shape == (nq, k) and sims.shape == (nq, k), what
    allowed = np.ones((nq, n), bool) if allowed is None else np.asarray(allowed, bool)
    m = allowed.sum(1)
    n_ret = np.minimum(m, k)
    slot = np.arange(k)[None, :]
    valid = slot < n_ret[:, None]
    # padding exactly where fewer than k rows are allowed: -1 / 0.0, and only at the end
    bad = np.argwhere(~valid & ((ids != -1) | (sims != 0)))
    assert bad.size == 0, f"{what}: padding expected at (query, slot) {bad[:5].tolist()}: {ids[tuple(bad[0])]}"
    rows = np.where(valid, ids - doc_base, -1)
    bad = np.argwhere(valid & ((rows < 0) | (rows >= n)))
    assert bad.size == 0, f"{what}: id out of range at {bad[:5].tolist()}: {ids[tuple(bad[0])]}"
    r0 = np.where(valid, rows, 0)
    bad = np.argwhere(valid & ~np.take_along_axis(allowed, r0, 1))
    assert bad.size == 0, f"{what}: a row the query may not return at {bad[:5].tolist()}"
    srt = np.sort(np.where(valid, rows, -1 - slot), axis=1)        # padding: distinct negatives
    dup = np.argwhere(srt[:, 1:] == srt[:, :-1])
    assert dup.size == 0, f"{what}: duplicate id in query {dup[0][0]}: {srt[dup[0][0]].tolist()}"
    # order (sim desc, id asc) among the returned rows
    both = valid[:, 1:]
    wrong = both & ((sims[:, 1:] > sims[:, :-1]) | ((sims[:, 1:] == sims[:, :-1]) & (rows[:, 1:] < rows[:, :-1])))
    bad = np.argwhere(wrong)
    assert bad.size == 0, f"{what}: order broken at (query, slot) {bad[:5].tolist()}"
    # each similarity within tol of the reference
    ref_r, tol_r = np.take_along_axis(ref, r0, 1), np.take_along_axis(tol, r0, 1)
    ratio = np.where(valid, np.abs(sims.astype(np.float64) - ref_r) / tol_r, 0.0)
    worst = float(ratio.max()) if ratio.size else 0.0
    i, j = np.unravel_index(int(ratio.argmax()), ratio.shape) if ratio.size else (0, 0)
    assert worst <= 1.0, (f"{what}: |sim - ref| / tol = {worst:.3g} at query {i} slot {j}: sim {sims[i, j]!r} "
                          f"ref {ref_r[i, j]!r} tol {tol_r[i, j]:.3g}")
    # the returned set against the reference k-th score (only queries with more than k allowed rows can differ)
    got = np.zeros((nq, n), bool)
    qi, sj = np.nonzero(valid)
    got[qi, rows[qi, sj]] = True
    full = m > k
    if full.any():
        refm = np.where(allowed[full], ref[full], -np.inf)
        kth = -np.partition(-refm, k - 1, axis=1)[:, k - 1]
        t2 = 2 * np.where(allowed[full], tol[full], 0.0).max(1)
        low = np.argwhere(valid[full] & (ref_r[full] < (kth - t2)[:, None]))
        assert low.size == 0, f"{what}: returned a row well below the k-th reference score (query {low[0][0]} of the full ones)"
        miss = np.argwhere((refm > (kth + t2)[:, None]) & ~got[full])
        assert miss.size == 0, f"{what}: missed row {miss[0][1]} well above the k-th reference score"
    short = ~full                                                # every allowed row comes back
    assert np.array_equal(got[short], allowed[short]), f"{what}: not every allowed row returned"
    return worst


def check_leading_ties(ids, tied, allowed, k, doc_base=0, what=""):
    """Rows tied[i] (bool [Q, N]) score exactly the same for query i and above every other allowed row: the answer
    starts with the allowed ones, lowest id first."""
    ids = np.asarray(ids, np.int64)
    for i in range(ids.shape[0]):
        want = np.flatnonzero(tied[i] & allowed[i])[:k]
        assert (ids[i, :want.size] - doc_base).tolist() == want.tolist(), f"{what}: tie order of query {i}"


def make_data(kind, n, d, nq, seed):
    """bf16 docs [n, d], queries [nq, d].  gauss: N(0, 1).  anti: docs <= 0 < queries elementwise, so every cosine is
    negative.  ortho: queries live (up to 1 %) in the first half of the dimensions, docs in the second, so every
    cosine is within about +-0.01 of 0, both signs.  zeros: anti plus zero rows (score 0, the best of every query)
    and a zero query (every score 0)."""
    g = torch.Generator().manual_seed(seed)
    x, q = torch.randn(n, d, generator=g), torch.randn(nq, d, generator=g)
    if kind in ("anti", "zeros"):
        x, q = -(x.abs() + 0.05), q.abs() + 0.05
    elif kind == "ortho":
        h = d // 2
        x[:, :h] *= 0.01
        q[:, h:] *= 0.01
    x, q = x.to(torch.bfloat16), q.to(torch.bfloat16)
    if kind == "zeros":
        x[torch.arange(0, n, 97)] = 0
        x[n - 1] = 0
        q[nq // 2] = 0
    return x, q


def report(what, worst):
    print(f"cosine-edges {what}: max |sim - ref| / tol = {worst:.4f}")


# (n_docs, d, nq, k, data, doc_base).  Sizes at +-1 of the 128-row CTA half, the 256-row tile, 64 tiles (one L2 window,
# 16384 rows) and one window + one tile (16640); d at +-8 of 64 and of 768 (the kernel switch), under one k-block, at
# and past 1024; nq at +-1 of 112 and of 224 and past two query blocks.  The reference work is nq * n * d <= 1e10.  At
# d > 1024 only Gaussian data: ordered or tied rows there would need the overflow fallback, which stops at 1024.
TOPK_CASES = [
    (1, 64, 1, 10, "gauss", 0),
    (7, 8, 111, 10, "gauss", BIG_BASE),
    (127, 16, 112, 255, "anti", 0),
    (128, 56, 113, 33, "ortho", BIG_BASE),
    (129, 72, 223, 256, "zeros", 0),
    (255, 760, 225, 10, "zeros", BIG_BASE),
    (257, 776, 449, 255, "gauss", 0),
    (16383, 768, 111, 10, "anti", 0),
    (16385, 64, 449, 1, "zeros", BIG_BASE),
    (16640, 1016, 225, 33, "gauss", 0),
    (16640, 1024, 224, 256, "ortho", BIG_BASE),
    (4097, 1032, 113, 10, "gauss", 0),
    (2000, 2056, 225, 33, "gauss", BIG_BASE),
    (16385, 256, 1, 256, "gauss", 0),
]


def _filter(n, nq, seed):
    """two random 30 % allow-lists; each query uses row 0, row 1 or none (-1)"""
    g = torch.Generator().manual_seed(seed)
    rows = torch.rand(2, n, generator=g) < 0.3
    qf = torch.randint(-1, 2, (nq,), generator=g)
    allowed = np.where(qf.numpy()[:, None] >= 0, rows.numpy()[qf.clamp(min=0).numpy()], True)
    return rows, qf, allowed


@gpu
@pytest.mark.parametrize("n,d,nq,k,kind,base", TOPK_CASES,
                         ids=[f"n{c[0]}-d{c[1]}-nq{c[2]}-k{c[3]}-{c[4]}" for c in TOPK_CASES])
def test_cosine_topk_edges(n, d, nq, k, kind, base):
    from document_retrieval_b200.cosine import CosineIndex, set_cosine_option
    seed = n * 7919 + d * 31 + nq
    docs, qs = make_data(kind, n, d, nq, seed)
    ref, tol = reference(docs, qs)
    frows, qf, allowed = _filter(n, nq, seed + 1)
    ix = CosineIndex(docs, doc_base=base)
    kernels = ["auto"] if d > 768 else ["auto", "mc"]          # d > 768: auto is the multicast kernel
    out = {}
    for kern in kernels:
        try:
            set_cosine_option("kernel", 1 if kern == "mc" else 0)
            out[kern] = ix.topk(qs, k), ix.topk(qs, k, doc_filter=frows, query_filter=qf)
        finally:
            set_cosine_option("kernel", 0)
    if kind == "zeros":                   # zero rows tie at 0 above every negative row; the zero query ties every row
        tied = np.repeat((docs == 0).all(1).numpy()[None, :], nq, 0)
        tied[nq // 2] = True
    for kern, ((ids, sims), (fids, fsims)) in out.items():
        what = f"{kern} n={n} d={d} nq={nq} k={k} {kind}"
        report(what, check_topk(ids.cpu(), sims.cpu(), ref, tol, k, doc_base=base, what=what))
        report(what + " filtered",
               check_topk(fids.cpu(), fsims.cpu(), ref, tol, k, allowed=allowed, doc_base=base, what=what + " filtered"))
        if kind == "zeros":
            check_leading_ties(ids.cpu(), tied, np.ones_like(tied), k, base, what)
            check_leading_ties(fids.cpu(), tied, allowed, k, base, what + " filtered")
    if "mc" in out:                                            # the two kernels are bit-identical (br_set_cosine_option)
        for a, b in zip(out["auto"], out["mc"]):
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@gpu
@pytest.mark.parametrize("kernel", ["auto", "mc"])
def test_cosine_exact_ties_below_the_overflow_cap(kernel):
    """40 bit-identical copies of one row, 3 in each of launches 1, 2 and 3 of the doubling schedule (tiles 0, 1-2,
    3-6) and 31 in launch 5 (tiles 15-30), at rows of both CTA halves and all four TMEM lane quarters of their tiles.
    No launch passes more than 1024 rows, so these queries go through the threshold path, not the exact fallback.  A
    query equal to the row must get the copies lowest id first with one identical similarity: at k = 10 the 9 copies
    of launches 1-3 and the first of launch 5, at k = 100 all 40 ahead of every other row.  (This assumes the UMMA
    accumulates identical rows at different M positions to identical fp32 values.)"""
    from document_retrieval_b200.cosine import CosineIndex, set_cosine_option
    n, d = 8192, 128
    g = torch.Generator().manual_seed(4242)
    docs = torch.randn(n, d, generator=g).to(torch.bfloat16)
    offs = [3, 100, 161, 230]                                  # quarters 0 and 3 of half 0, 1 and 3 of half 1
    pos = [0 * 256 + 3, 0 * 256 + 161, 0 * 256 + 230,          # launch 1: tile 0
           1 * 256 + 100, 2 * 256 + 3, 2 * 256 + 230,          # launch 2: tiles 1-2
           3 * 256 + 161, 5 * 256 + 100, 6 * 256 + 3]          # launch 3: tiles 3-6
    pos += [t * 256 + offs[(t + j) % 4] + 8 * j for t in range(15, 31) for j in range(2)][:31]   # launch 5
    pos = np.sort(np.asarray(pos))
    assert pos.size == 40 and np.unique(pos).size == 40
    src = docs[pos[0]].clone()
    docs[torch.from_numpy(pos)] = src
    qs = torch.randn(300, d, generator=g).to(torch.bfloat16)
    qs[0] = src                                                # query columns 0 and 150: both halves of the query block
    qs[150] = src
    ref, tol = reference(docs, qs)
    ix = CosineIndex(docs)
    try:
        set_cosine_option("kernel", 1 if kernel == "mc" else 0)
        for k in (10, 100):
            ids, sims = ix.topk(qs, k)
            ids, sims = ids.cpu().numpy(), sims.cpu().numpy()
            for qi in (0, 150):
                c = min(k, 40)
                assert ids[qi, :c].tolist() == pos[:c].tolist(), (k, qi, ids[qi, :c])
                assert (sims[qi, :c] == sims[qi, 0]).all(), (k, qi, sims[qi, :c])
                assert (sims[qi, c:] < sims[qi, 0]).all()
            report(f"ties {kernel} k={k}", check_topk(ids, sims, ref, tol, k, what=f"ties {kernel} k={k}"))
    finally:
        set_cosine_option("kernel", 0)


def _rerank_null_norms(ix, qs, cand, k):
    """br_cosine_rerank through the C ABI with doc_inv_norm_dev = NULL (norms computed in the gather kernel)"""
    from document_retrieval_b200 import _lib
    lib = _lib.load()
    q = qs.to(ix.device).contiguous()
    cd = cand.to(device=ix.device, dtype=torch.int32).contiguous()
    nq, c = cd.shape
    ids = torch.empty((nq, k), dtype=torch.int32, device=ix.device)
    sims = torch.empty((nq, k), dtype=torch.float32, device=ix.device)
    _lib.check(lib.br_cosine_rerank(_lib.ptr(ix.docs), None, ix.n_docs, ix.dim, _lib.ptr(q), nq, _lib.ptr(cd), c, k,
                                    _lib.ptr(ids), _lib.ptr(sims), C.c_void_p(_lib.stream_ptr(ix.device))),
               "br_cosine_rerank")
    return ids, sims


def _candidates(n, nq, c, seed):
    """[nq, c] random rows with repeats; -1 slots at the start, middle and end of some rows; one row all -1"""
    g = torch.Generator().manual_seed(seed)
    cand = torch.randint(0, n, (nq, c), generator=g, dtype=torch.int32)
    if c >= 3:
        cand[1, 0] = cand[2, c // 2] = cand[3, c - 1] = -1
        cand[4, :: 3] = -1
    cand[nq - 1] = -1
    if c >= 2:
        cand[5, 1] = cand[5, 0]                                # a repeated candidate
    return cand


# (d, c, k): NV = ceil(d / 256) 16-byte vectors per lane from 1 to 4, full (256, 512, 768, 1024) and partial last
# vectors (8: lane 0 only, 248, 264: lane 0 only, 520, 776); c around the 2048-entry rounds of the final selection and
# not a multiple of 4 or 32; k > c; k = 1024.
RERANK_CASES = [(8, 1, 1), (248, 3, 10), (256, 5, 1024), (264, 33, 10), (512, 2047, 1024), (520, 2049, 10),
                (768, 5000, 1024), (776, 33, 1), (1024, 2049, 1024), (264, 5000, 10)]


@gpu
@pytest.mark.parametrize("d,c,k", RERANK_CASES, ids=[f"d{x[0]}-c{x[1]}-k{x[2]}" for x in RERANK_CASES])
def test_cosine_rerank_edges(d, c, k):
    from document_retrieval_b200.cosine import CosineIndex
    n, nq = 3000, 8
    seed = d * 131 + c
    docs, qs = make_data("gauss", n, d, nq, seed)
    docs[torch.arange(0, n, 50)] = 0                           # zero rows score 0
    qs[6] = 0                                                  # a zero query: every candidate scores 0, ties by id
    cand = _candidates(n, nq, c, seed)
    ref, tol = reference(docs, qs)
    allowed = np.zeros((nq, n), bool)
    cn = cand.numpy()
    for i in range(nq):
        allowed[i, cn[i][cn[i] >= 0]] = True
    ix = CosineIndex(docs)
    ids, sims = ix.rerank(qs, cand, k)
    assert ids.dtype == torch.int32 and ids.shape == (nq, k)
    what = f"rerank d={d} c={c} k={k}"
    report(what, check_topk(ids.cpu().numpy().astype(np.int64), sims.cpu(), ref, tol, k, allowed=allowed, what=what))
    check_leading_ties(ids.cpu()[6:7], np.ones((1, n), bool), allowed[6:7], k, what=what)
    # k_cosine_rerank accumulates ||x||^2 with the lane order, fmaf chain and butterfly of k_row_inv_norm
    ids0, sims0 = _rerank_null_norms(ix, qs, cand, k)
    assert torch.equal(ids0, ids) and torch.equal(sims0, sims)


@gpu
def test_cosine_empty_batch():
    """nq = 0 returns empty results.  (Fixed: an empty batch failed the null-pointer check, as torch's empty tensors
    have data_ptr 0.)"""
    from document_retrieval_b200.cosine import CosineIndex
    docs, qs = make_data("gauss", 100, 64, 3, 11)
    ix = CosineIndex(docs)
    cand = torch.zeros((0, 5), dtype=torch.int32)
    for ids, sims in (ix.rerank(qs[:0], cand, 10), _rerank_null_norms(ix, qs[:0], cand, 10), ix.topk(qs[:0], 10),
                      ix.topk(qs[:0], 10, doc_filter=torch.ones(100, dtype=torch.bool))):
        assert ids.shape == (0, 10) and sims.shape == (0, 10)


@gpu
@pytest.mark.parametrize("bad_id", ["n_docs", 2 ** 31 - 1, -2])
def test_cosine_rerank_rejects_out_of_range_ids(bad_id):
    """A candidate id outside [-1, n_docs) is BR_ERR_INVALID.  It used to score -inf and come back as a row that does
    not exist (k >= c here, so it would be returned)."""
    from document_retrieval_b200._lib import BRError
    from document_retrieval_b200.cosine import CosineIndex
    n = 300
    docs, qs = make_data("gauss", n, 128, 4, 12)
    ix = CosineIndex(docs)
    bad = n if bad_id == "n_docs" else bad_id
    cand = torch.tensor([[0, 5, -1, 7], [1, 2, 3, 4], [9, bad, 8, -1], [-1, -1, -1, -1]], dtype=torch.int32)
    with pytest.raises(BRError, match=r"outside \[-1, n_docs\)"):
        ix.rerank(qs, cand, 4)
    with pytest.raises(BRError, match=r"outside \[-1, n_docs\)"):
        _rerank_null_norms(ix, qs, cand, 4)
    cand[2, 1] = n - 1                                         # the flag belongs to one call
    ids, _ = ix.rerank(qs, cand, 4)
    assert sorted(ids[2].tolist()) == [-1, 8, 9, n - 1]


@pytest.mark.parametrize("d", [8, 64, 776, 2056])
@pytest.mark.parametrize("kind", ["gauss", "anti", "ortho", "zeros"])
def test_reference_and_bound_cover_torch_fp32(kind, d):
    """CPU: the float64 reference with its tolerance bounds torch's fp32 normalise + matmul, and check_topk accepts
    that restatement's answer and rejects a broken copy of it."""
    n, nq, k = 700, 40, 20
    docs, qs = make_data(kind, n, d, nq, d + len(kind))
    ref, tol = reference(docs, qs)
    ids, sims = orc.cosine_topk(docs.float().numpy(), qs.float().numpy(), n)
    full = np.empty((nq, n), np.float32)
    np.put_along_axis(full, ids, sims, 1)
    ratio = np.abs(full - ref) / tol
    assert ratio.max() <= 1.0, (kind, d, ratio.max())
    worst = check_topk(ids[:, :k], sims[:, :k], ref, tol, k, what=f"torch fp32 {kind} d={d}")
    assert worst <= 1.0
    shifted = ids[:, :k].copy()
    shifted[3, 0] = (shifted[3, 0] + 256) % n                  # a row shifted by one tile
    with pytest.raises(AssertionError):
        check_topk(shifted, sims[:, :k], ref, tol, k)
    padded = ids[:, :k].copy()
    padded[5, k - 1] = -1                                      # padding where k rows are allowed
    with pytest.raises(AssertionError):
        check_topk(padded, sims[:, :k], ref, tol, k)
