"""Corpus sharding across GPUs: one process per GPU, contiguous row ranges, replicated queries.

Every rank runs the search pipeline on its own shard against ONE global per-query threshold
(``engine.search_shards``): two small ``all_gather`` s of per-shard order statistics (the top-J sample scores,
then the exact scores of every shard's best few candidates -- the pilot of the two-round rescore; ~2-3 MB per rank
at 8192 queries) make every shard append and rescore only its share of the candidates, and ONE ``all_gather`` of a
packed block per rank (``[nq, k]`` exact scores, global rows, overflow flags) over NCCL / NVLink followed by the
G-way merge kernel (K3) gives every rank the certified global top-k.  No collective needs the host: the error
bound lives on the device and the certificate is read back asynchronously.  Exact
fp64 scores are comparable across shards, so the merge is exact.  The reference has no multi-GPU path for this
stage (SURVEY.md section 2.4); this is the design of section 8e.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def shard_range(n_total, world_size, rank):
    """Contiguous, balanced row range ``[lo, hi)`` of ``rank`` (first ``n_total % world_size`` ranks get one more)."""
    base, rem = divmod(int(n_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class GroupComm:
    """The collectives ``engine.search_shards`` needs, over a ``torch.distributed`` group (nccl or gloo)."""

    def __init__(self, group=None):
        self.group = group
        self.world = dist.get_world_size(group)

    def gather(self, t):
        """``t`` (same shape on every rank) -> ``[world, *t.shape]`` on every rank: ONE collective straight into the
        result (no per-rank list, no ``torch.stack`` copy)."""
        t = t.contiguous()
        out = torch.empty((self.world * t.numel(),), dtype=t.dtype, device=t.device)
        dist.all_gather_into_tensor(out, t.reshape(-1), group=self.group)
        return out.view((self.world,) + tuple(t.shape))

    def max_(self, t):
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return t

    def sum_(self, t):
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def sum_int(self, v):
        dev = "cuda" if dist.get_backend(self.group) == "nccl" else "cpu"
        t = torch.tensor([int(v)], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return int(t.item())


def upload_rows(host_rows, group=None, device=None):
    """Host -> device copy of a row batch that every rank holds on the host (the query batch of a serving step):
    each rank copies only ITS slice over PCIe and the slices are all-gathered over NVLink, so the node moves the
    batch across PCIe once instead of once per GPU (8 x 64 MB per step at 8192 x 2048 fp32 otherwise).
    Returns the full ``[n, d]`` device tensor on every rank."""
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return host_rows.to(device, non_blocking=True)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n = host_rows.shape[0]
    per = (n + world - 1) // world
    lo, hi = min(n, rank * per), min(n, (rank + 1) * per)
    full = torch.empty((world * per,) + tuple(host_rows.shape[1:]), dtype=host_rows.dtype, device=device)
    mine = torch.zeros((per,) + tuple(host_rows.shape[1:]), dtype=host_rows.dtype, device=device)
    if hi > lo:
        mine[: hi - lo].copy_(host_rows[lo:hi], non_blocking=True)
    parts = list(full.view((world, per) + tuple(host_rows.shape[1:])).unbind(0))
    dist.all_gather(parts, mine, group=group)
    return full[:n]


def gather_topk(scores, idx, group=None):
    """all_gather of local ``[nq, k]`` results -> ``[G, nq, k]`` on every rank (works on gloo and nccl)."""
    world = dist.get_world_size(group)
    s_all = [torch.empty_like(scores) for _ in range(world)]
    i_all = [torch.empty_like(idx) for _ in range(world)]
    dist.all_gather(s_all, scores.contiguous(), group=group)
    dist.all_gather(i_all, idx.contiguous(), group=group)
    return torch.stack(s_all), torch.stack(i_all)


def merge_reference(scores, idx, k):
    """Host/torch statement of the merge rule (score desc, index asc) used to test the K3 kernel and the
    gloo path: ``scores/idx [G, nq, kk]`` -> ``[nq, k]``."""
    g, nq, kk = scores.shape
    s = scores.permute(1, 0, 2).reshape(nq, g * kk)
    i = idx.permute(1, 0, 2).reshape(nq, g * kk)
    big = torch.iinfo(torch.int64).max
    i_key = torch.where(i < 0, torch.full_like(i, big), i)
    order = torch.argsort(i_key, dim=1, stable=True)
    s, i = torch.gather(s, 1, order), torch.gather(i, 1, order)
    order = torch.argsort(s, dim=1, descending=True, stable=True)
    return torch.gather(s, 1, order)[:, :k], torch.gather(i, 1, order)[:, :k]


def sharded_search(store, queries, k, group=None, n_total=None, **kw):
    """Search the corpus whose rows are sharded over the ranks of ``group``; every rank passes the same queries
    and gets the same global ``(scores, idx)``.  ``n_total`` (the global row count) saves one tiny all-reduce."""
    from .engine import search_shards
    stores = list(store) if isinstance(store, (list, tuple)) else [store]
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return search_shards(stores, queries, k, **kw)
    return search_shards(stores, queries, k, comm=GroupComm(group), n_total=n_total, **kw)


def sharded_range_search(store, queries, min_score, group=None, **kw):
    """Range search (``engine.range_search_shards``) over the corpus whose rows are sharded over the ranks of
    ``group``; every rank passes the same queries and gets the same global ``RangeResult``."""
    from .engine import range_search_shards
    stores = list(store) if isinstance(store, (list, tuple)) else [store]
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return range_search_shards(stores, queries, min_score, **kw)
    return range_search_shards(stores, queries, min_score, comm=GroupComm(group), **kw)


def sharded_range_count(store, queries, min_score, group=None, **kw):
    """``engine.range_count_shards`` over the ranks of ``group``: the global length of every range-search list."""
    from .engine import range_count_shards
    stores = list(store) if isinstance(store, (list, tuple)) else [store]
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return range_count_shards(stores, queries, min_score, **kw)
    return range_count_shards(stores, queries, min_score, comm=GroupComm(group), **kw)


def sharded_similar_pairs(store, min_score, group=None, **kw):
    """Similar pairs (``engine.similar_pairs_shards``) of the corpus whose rows are sharded over the ranks of ``group``:
    every pair of rows ``i < j`` scoring at least ``min_score``, each once; every rank gets the same ``RangeResult``."""
    from .engine import similar_pairs_shards
    stores = list(store) if isinstance(store, (list, tuple)) else [store]
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return similar_pairs_shards(stores, min_score, **kw)
    return similar_pairs_shards(stores, min_score, comm=GroupComm(group), **kw)
