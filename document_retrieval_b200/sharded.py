"""Doc-sharded BM25 across the GPUs of one box (one process per GPU, torch.distributed).

The reference is single-process; sharding follows SURVEY 8e: contiguous doc ranges per rank, the
corpus statistics (N, sum of doc lengths, df histogram) all-reduced once at build time so that
every shard computes bit-identical idf / avgdl, and at query time only each rank's [Q, k]
(global id, float64 score) candidates cross NVLink (all-gather) before the k*G -> k merge.
Top-k over a doc partition is exactly decomposable, so sharded results equal single-GPU results
bit for bit.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from ._lib import check, ptr


def shard_bounds(n_docs: int, world: int):
    """Contiguous doc ranges: shard r = [r*ceil(N/G), min(N, (r+1)*ceil(N/G)))."""
    per = -(-n_docs // world)
    return [(min(n_docs, r * per), min(n_docs, (r + 1) * per)) for r in range(world)]


def group_shard_bounds(row_group, world: int):
    """Contiguous row ranges that never split a group: the cuts of ``shard_bounds`` moved forward to the next group
    start.  ``row_group`` is the non-decreasing row -> group map of the whole corpus.  A shard may come out empty when
    one group spans more than a shard's share of the rows."""
    rg = np.asarray(torch.as_tensor(row_group).cpu())
    n = rg.shape[0]
    starts = np.flatnonzero(np.r_[True, rg[1:] != rg[:-1]]) if n else np.zeros(0, np.int64)
    starts = np.r_[starts, n]
    cuts = [0] + [int(starts[np.searchsorted(starts, lo)]) for lo, _ in shard_bounds(n, world)[1:]] + [n]
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def reduce_stats(local_df: torch.Tensor, n_docs: int, sum_dl: int, group=None):
    """All-reduce (sum) of the df histogram and (N, sum dl) -> (df int64[V] on host, N, sum_dl)."""
    df = local_df.to(torch.int64)
    st = torch.tensor([n_docs, sum_dl], dtype=torch.int64, device=df.device)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(df, group=group)
        dist.all_reduce(st, group=group)
    st = st.cpu()
    return df.cpu().numpy(), int(st[0]), int(st[1])


def pack_records(ids: torch.Tensor, scores: torch.Tensor):
    """[Q, k] (int64 global id, float64 score) -> int64[Q, k, 2] records (the score's bits in [..., 1])."""
    return torch.stack([ids.to(torch.int64), scores.to(torch.float64).view(torch.int64)], dim=-1).contiguous()


def gather_records(rec: torch.Tensor, group=None):
    """ONE all-gather of the per-rank packed [Q, k, 2] records -> [G, Q, k, 2]."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return rec[None]
    out = torch.empty((world * rec.shape[0],) + tuple(rec.shape[1:]), dtype=rec.dtype, device=rec.device)
    dist.all_gather_into_tensor(out, rec.contiguous(), group=group)
    return out.view((world,) + tuple(rec.shape))


def gather_candidates(ids: torch.Tensor, scores: torch.Tensor, group=None):
    """all-gather of per-rank [Q, k] candidates -> ([G, Q, k] ids, [G, Q, k] scores), one collective."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return ids[None], scores[None]
    allr = gather_records(pack_records(ids, scores), group)
    return allr[..., 0].contiguous(), allr[..., 1].contiguous().view(torch.float64)


def merge_records_cuda(all_rec: torch.Tensor, k: int):
    """br_topk_merge_records: packed records [G, Q, k, 2] -> ([Q, k] ids, [Q, k] scores) by (score desc, id asc)."""
    lib = _lib.load()
    g, q, kk, _ = all_rec.shape
    dev = all_rec.device
    if kk != k:
        raise ValueError("candidate width must equal k")
    out_ids = torch.empty((q, k), dtype=torch.int64, device=dev)
    out_sc = torch.empty((q, k), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        check(lib.br_topk_merge_records(ptr(all_rec.contiguous()), g, q, k, ptr(out_ids), ptr(out_sc), _lib.stream_ptr(dev)),
              "br_topk_merge_records")
    return out_ids, out_sc


def merge_topk_cuda(all_ids: torch.Tensor, all_sc: torch.Tensor, k: int):
    """br_topk_merge: [G, Q, k] -> [Q, k] by (score desc, id asc)."""
    lib = _lib.load()
    g, q, kk = all_ids.shape
    dev = all_ids.device
    out_ids = torch.empty((q, k), dtype=torch.int64, device=dev)
    out_sc = torch.empty((q, k), dtype=torch.float64, device=dev)
    if kk != k:
        raise ValueError("candidate width must equal k")
    with torch.cuda.device(dev):
        check(lib.br_topk_merge(ptr(all_ids.contiguous()), ptr(all_sc.contiguous()), g, q, k, ptr(out_ids), ptr(out_sc),
                                _lib.stream_ptr(dev)), "br_topk_merge")
    return out_ids, out_sc


def local_filter_slice(doc_filter, lo: int, n_local: int):
    """A filter over GLOBAL doc ids (bool [N] or [F, N]) -> this shard's columns [lo, lo + n_local)."""
    if doc_filter is None:
        return None
    f = torch.as_tensor(doc_filter)
    if f.dtype != torch.bool or f.dim() not in (1, 2) or f.shape[-1] < lo + n_local:
        raise ValueError("doc_filter must be a bool array [N] or [F, N] over the global doc ids")
    return f[..., lo:lo + n_local]


def local_group_candidates(candidate_groups, group_base: int, n_groups: int):
    """GLOBAL candidate group ids [Q, c] (-1 = empty) -> this shard's local ids: ids in [group_base, group_base + n_groups)
    minus group_base, every other id -1.  -> (local int32 [Q, c], number of ids this shard owns)."""
    g = torch.as_tensor(candidate_groups).to(torch.int64)
    own = (g >= group_base) & (g < group_base + n_groups)
    return torch.where(own, g - group_base, torch.full_like(g, -1)).to(torch.int32), int(own.sum())


class ShardedBM25:
    """One rank's view of a doc-sharded index.  ``local`` is this rank's ``BM25`` shard (built with
    ``doc_base`` = first global doc id of the shard and the all-reduced statistics)."""

    def __init__(self, local, group=None, merge=merge_topk_cuda, share_thresholds=True):
        self.local, self.group, self.merge = local, group, merge
        self.share_thresholds = share_thresholds
        self._xr = {}                    # k -> exchange rounds agreed between the ranks (-1: off)
        self._cb = None
        self._thr_views = {}

    # ---- threshold sharing (br_set_thr_exchange): every shard prunes with a bound learnt on the WHOLE corpus.  The library
    # hands over its thresholds (after seeding) or its current k best scores per query (after a tile launch); this callback
    # all-gathers them over the shards on the current stream and the library takes the maximum / the k-th largest of the
    # union - the threshold a single index would have after the same fraction of its docs.
    def _exchange(self, local_ptr, gathered_ptr, n_floats, stream, user):
        try:
            world = dist.get_world_size(self.group)
            key = (local_ptr, gathered_ptr, n_floats)
            view = self._thr_views.get(key)
            if view is None:
                def wrap(ptr, n):
                    class _Arr:
                        __cuda_array_interface__ = {"shape": (n,), "typestr": "<f4", "data": (ptr, False), "version": 3}
                    return torch.as_tensor(_Arr(), device=self.local._device)
                view = (wrap(local_ptr, n_floats), wrap(gathered_ptr, n_floats * world))
                self._thr_views[key] = view
            dist.all_gather_into_tensor(view[1], view[0], group=self.group)     # on the current stream
            return 0
        except Exception:                # never raise through the C frame
            import traceback
            traceback.print_exc()
            return -1

    def _setup_exchange(self, k):
        """Agree on the number of exchanges per batch (same on every rank, or none at all) for this k."""
        if k in self._xr:
            return self._xr[k]
        rounds = -1
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if (self.share_thresholds and world > 1 and hasattr(self.local, "_h") and self.local._h is not None
                and self.merge is merge_topk_cuda):
            lib = _lib.load()
            n = int(lib.br_tile_launch_count(self.local._h, int(k)))
            t = torch.tensor([n], dtype=torch.int64, device=self.local._device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN, group=self.group)
            rounds = int(t.item()) - 1 if int(t.item()) > 0 else -1
        self._xr[k] = rounds
        return rounds

    def _set_exchange(self, rounds):
        lib = _lib.load()
        if rounds >= 0:
            if self._cb is None:
                self._cb = _lib.THR_EXCHANGE_FN(self._exchange)
            check(lib.br_set_thr_exchange(self.local._h, self._cb, None, int(rounds), dist.get_world_size(self.group)), "br_set_thr_exchange")
        else:
            check(lib.br_set_thr_exchange(self.local._h, None, None, -1, 1), "br_set_thr_exchange")

    @classmethod
    def from_local_token_ids(cls, doc_offsets, token_ids, vocab_size, doc_base, k1=1.5, b=0.75, *,
                             variant="notebook", dedup_query=None, device=None, group=None):
        from .bm25 import BM25
        m = BM25.from_token_ids(doc_offsets, token_ids, vocab_size, k1, b, variant=variant, dedup_query=dedup_query,
                                device=device, doc_base=doc_base, finalize=False)
        st = m.stats()
        df, n_stat, sum_dl = reduce_stats(m.local_df_tensor(), st["n_docs"], st["sum_dl"], group)
        m.finalize(n_stat, sum_dl, df)
        self = cls(m, group)
        self.n_docs_global = n_stat
        return self

    def retrieve_top_n_batch(self, queries, n=10, doc_filter=None, query_filter=None):
        """-> (global ids int64[Q, n], float64 scores[Q, n]) identical on every rank.  ``doc_filter``: bool [N] or
        [F, N] over the GLOBAL doc ids (with ``query_filter`` int [Q] for [F, N]); each rank uses its own columns."""
        fkw = {}
        if doc_filter is not None or query_filter is not None:
            fkw = dict(doc_filter=local_filter_slice(doc_filter, self.local.doc_base, self.local.corpus_size),
                       query_filter=query_filter)
        if hasattr(self.local, "retrieve_records_batch") and self.merge is merge_topk_cuda:
            # CUDA shard: the library emits packed {global id, score} records - one all-gather, merged straight from
            # the gathered buffer
            rounds = self._setup_exchange(n)
            if rounds >= 0:
                self._set_exchange(rounds)
            try:
                rec = self.local.retrieve_records_batch(queries, n, **fkw)
            finally:
                if rounds >= 0:
                    self._set_exchange(-1)
            allr = gather_records(rec, self.group)
            if allr.shape[0] == 1:
                return rec[..., 0].contiguous(), rec[..., 1].contiguous().view(torch.float64)
            ids, sc = merge_records_cuda(allr, n)
            if rounds >= 0:
                # with shared thresholds a query that has fewer than n matching docs in the WHOLE corpus comes back short:
                # those (rare) queries are repeated with local thresholds, whose zero-score fill is exact.  A filtered
                # query can return at most as many docs as its filter allows, so "short" is measured against that.
                total = getattr(self, "n_docs_global", None) or n
                need = torch.full((ids.shape[0],), min(n, total), dtype=torch.int64, device=ids.device)
                if fkw:
                    f = torch.as_tensor(doc_filter)
                    allowed = f.to(ids.device).reshape(-1, f.shape[-1]).sum(-1)          # [F] allowed docs per row
                    if query_filter is None:
                        need = torch.clamp(need, max=int(allowed[0]))
                    else:
                        qf = torch.as_tensor(query_filter).to(device=ids.device, dtype=torch.int64)
                        per_q = torch.where(qf >= 0, allowed[qf.clamp(min=0, max=allowed.numel() - 1)], need)
                        need = torch.minimum(need, per_q)
                last = ids.gather(1, (need - 1).clamp(min=0)[:, None])[:, 0]
                short = torch.nonzero((need > 0) & (last < 0)).flatten()
                if short.numel():
                    q_terms, q_off = self.local.pack_queries(queries)
                    q_terms, q_off = q_terms.cpu(), q_off.cpu()
                    rows = short.cpu().tolist()
                    sub_t = torch.cat([q_terms[int(q_off[r]):int(q_off[r + 1])] for r in rows]) if rows else q_terms[:0]
                    sub_o = torch.tensor([0] + [int(q_off[r + 1] - q_off[r]) for r in rows], dtype=torch.int32).cumsum(0).to(torch.int32)
                    sub_kw = dict(fkw)
                    if fkw and query_filter is not None:
                        sub_kw["query_filter"] = torch.as_tensor(query_filter)[short.cpu()]
                    rec2 = self.local.retrieve_records_batch((sub_t.to(torch.int32), sub_o), n, **sub_kw)
                    i2, s2 = merge_records_cuda(gather_records(rec2, self.group), n)
                    ids[short], sc[short] = i2, s2
            return ids, sc
        ids, sc = self.local.retrieve_top_n_batch(queries, n, **fkw)
        gids = torch.where(ids >= 0, ids.to(torch.int64) + self.local.doc_base, torch.full_like(ids, -1, dtype=torch.int64))
        all_ids, all_sc = gather_candidates(gids, sc, self.group)
        if all_ids.shape[0] == 1:
            return gids, sc
        return self.merge(all_ids, all_sc, n)


class ShardedCosineIndex:
    """Row-sharded brute-force cosine top-k (BASELINE config 5: 10 M x 768 bf16 over 8 GPUs; the
    reference's single-process path is team_run1.py:269-282).  Each rank holds the embedding rows
    ``[row_base, row_base + n_local)``, queries are replicated (10 k x 768 x 2 B = 15 MB), every rank
    runs the fused GEMM + top-k on its rows and only the [Q, k] (global row, cosine) candidates are
    all-gathered and merged - bit-identical to the single-GPU result because top-k over a row
    partition is exactly decomposable and ties break on the global row id.

    ``row_group`` (optional): the GLOBAL group (document) id of each local row, non-decreasing, for ``topk_groups``.
    Every rank must hold whole groups (split with ``group_shard_bounds``); the local index numbers its groups from the
    rank's first group, which it adds back to the ids it returns.  ``n_groups``: the global group id bound of this rank
    (default: its largest group + 1)."""

    def __init__(self, local_embeddings, row_base, device=None, group=None, merge=merge_topk_cuda, local=None,
                 row_group=None, n_groups=None):
        if local is None:
            from .cosine import CosineIndex
            gkw = {}
            if row_group is not None:
                rg = torch.as_tensor(row_group).to(torch.int64)
                g_lo = int(rg.min()) if rg.numel() else 0
                hi = int(n_groups) if n_groups is not None else (int(rg.max()) + 1 if rg.numel() else 1)
                gkw = dict(row_group=rg - g_lo, n_groups=hi - g_lo, group_base=g_lo)
            local = CosineIndex(local_embeddings, device=device, doc_base=row_base, **gkw)
        self.local, self.group, self.merge = local, group, merge

    def topk(self, query_embeddings, k=10, doc_filter=None, query_filter=None):
        """-> (global rows int64[Q, k], cosine float64[Q, k] (fp32 values widened)) on every rank.  ``doc_filter``: bool
        [N] or [F, N] over the GLOBAL rows (with ``query_filter`` int [Q] for [F, N]); each rank uses its own columns."""
        fkw = {}
        if doc_filter is not None or query_filter is not None:
            fkw = dict(doc_filter=local_filter_slice(doc_filter, self.local.doc_base, self.local.n_docs),
                       query_filter=query_filter)
        ids, sims = self.local.topk(query_embeddings, k, **fkw)
        return self._merge(ids, sims, k)

    def topk_groups(self, query_embeddings, k=10, doc_filter=None, query_filter=None):
        """Group-level top-k (``CosineIndex.topk_groups``) over all ranks -> (global group ids int64[Q, k], cosine
        float64[Q, k]) on every rank, identical to one index over all rows.  ``doc_filter``: bool [G] or [F, G] over
        the GLOBAL group ids (with ``query_filter`` int [Q] for [F, G]); each rank uses its own columns."""
        fkw = {}
        if doc_filter is not None or query_filter is not None:
            fkw = dict(doc_filter=local_filter_slice(doc_filter, self.local.group_base, self.local.n_groups),
                       query_filter=query_filter)
        ids, sims = self.local.topk_groups(query_embeddings, k, **fkw)
        return self._merge(ids, sims, k)

    def rerank_groups(self, query_embeddings, candidate_groups, k=10):
        """Grouped re-rank (``CosineIndex.rerank_groups``) of candidate groups [Q, c] given as GLOBAL group ids (-1 =
        empty), the same on every rank -> (global group ids int64[Q, k], cosine float64[Q, k]) on every rank, identical
        to one index over all rows.  Rank r owns the ids [group_base, group_base + n_groups) of its local index; an id
        below -1 or owned by no rank raises ValueError on every rank."""
        cand = torch.as_tensor(candidate_groups).to(device=self.local.device, dtype=torch.int64)
        if bool((cand < -1).any()):
            raise ValueError("candidate group ids must be >= -1")
        local, owned = local_group_candidates(cand, self.local.group_base, self.local.n_groups)
        t = torch.tensor([owned], dtype=torch.int64, device=cand.device)
        if dist.is_initialized() and dist.get_world_size(self.group) > 1:
            dist.all_reduce(t, group=self.group)
        if int(t) != int((cand >= 0).sum()):
            raise ValueError("a candidate group id is owned by no rank")
        ids, sims = self.local.rerank_groups(query_embeddings, local, k)
        ids = torch.where(ids >= 0, ids.to(torch.int64) + self.local.group_base, torch.full_like(ids, -1, dtype=torch.int64))
        return self._merge(ids, sims, k)

    def _merge(self, ids, sims, k):
        sims = sims.to(torch.float64)
        all_ids, all_sc = gather_candidates(ids, sims, self.group)
        if all_ids.shape[0] == 1:
            return ids, sims
        return self.merge(all_ids, all_sc, k)
