"""Filtered search (``label_mask``) through the multi-rank pipeline on CPU: two gloo ranks, each with a CPU model shard
with row labels (its ``_label_counts``, and ``_eligible``, through which the model's ``_filter``, ``_sample`` and
``_exact_small`` apply them).  Covers the globally reduced label histogram and eligible counts, the sharded
threshold over masked samples, the routing of rows with few eligible rows to thr = -inf and the certificate of their
short lists, the re-run loop, and the small-corpus branch -- each against the full-corpus fp64 model restricted to the
eligible rows.  The labelled kernels themselves are tested on the B200 (test_gpu_filtered_search.py)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _allowed(masks, labels):
    """[nq, n] bool: bit labels[v] of masks[q] is set."""
    return torch.bitwise_and(torch.bitwise_right_shift(masks[:, None], labels[None, :]), 1) != 0


def _labelled_shard_class():
    import cpu_model

    class LabelledShard(cpu_model.ModelShard):
        def __init__(self, rows, dims, labels, index_offset=0):
            super().__init__(rows, dims, index_offset)
            self.labels = labels.long()
            self.label_version = 0

        def _label_counts(self):
            return torch.bincount(self.labels, minlength=64)

        def set_labels(self, ids, labels):
            """CorpusStore.set_labels: a collective call, every shard applies its own rows of the same arguments."""
            loc = torch.as_tensor(ids) - self.index_offset
            mine = (loc >= 0) & (loc < self.n)
            self.labels[loc[mine]] = torch.as_tensor(labels)[mine]
            self.label_version += 1

        def _eligible(self, label_mask, step=1):
            return None if label_mask is None else _allowed(label_mask, self.labels[::step])

    return LabelledShard


def _worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cross_modal_video_engine_b200 import distributed, engine
    import cpu_model
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cpu_model.patch_engine(setattr)
    LabelledShard = _labelled_shard_class()
    nv, nq, d, k = 40000, 14, 32, 20
    g = torch.Generator().manual_seed(11)
    V, Q = torch.randn((nv, d), generator=g), torch.randn((nq, d), generator=g)
    labels = torch.randint(0, 62, (nv,), generator=g)
    labels[torch.randperm(nv, generator=g)[:3000]] = 63        # 3 000 rows: more than the lists hold at first
    labels[torch.randperm(nv, generator=g)[:5]] = 62           # a label with fewer rows than k
    for qi in range(nq):                                        # planted neighbours
        rows = torch.randperm(nv, generator=g)[:25]
        V[rows] = Q[qi] + 0.3 * torch.randn((25, d), generator=g)
    dense = torch.nonzero(labels == 63).flatten()               # query 1: every label-63 row is a near neighbour
    V[dense] = Q[1] * 2.0 + 0.4 * torch.randn((len(dense), d), generator=g)
    for qi in (7,):                                             # dense, unfiltered-sized neighbourhood
        rows = torch.randperm(nv, generator=g)[:6000]
        V[rows] = Q[qi] * 2.0 + 0.4 * torch.randn((6000, d), generator=g)
    bit = lambda ls: sum(1 << l for l in ls)                    # noqa: E731
    masks = [-1, bit([63]), bit([5]), 0, bit([62]), bit([62, 7]), bit(range(0, 64, 4)), bit(range(16)),
             bit([1, 2, 3]), -1, bit(range(32, 64)), bit([63, 0]), bit([9]) | (1 << 63), bit(range(8, 40))]
    masks = torch.tensor([m - (1 << 64) if m >= (1 << 63) else m for m in masks], dtype=torch.int64)
    excl = torch.full((nq,), -1, dtype=torch.int64)
    excl[5] = int(torch.nonzero(labels == 62).flatten()[0])    # excluding one of a short list's rows
    excl[9] = 17
    lo, hi = distributed.shard_range(nv, world, rank)
    shard = LabelledShard(V[lo:hi], (d,), labels[lo:hi], index_offset=lo)
    full = cpu_model.ModelShard(V, (d,))
    _, qr, qn, _, _ = full.prepare_queries(Q, [1.0])
    exact = full._exact(qr, qn, [1.0])
    exact_m = exact.clone()
    exact_m[~_allowed(masks, labels)] = float("-inf")

    def check(s, i, kk, ex=None):
        bad = []
        for r in range(nq):
            want_s, want_i, _ = cpu_model._sorted_topk(exact_m[r], torch.arange(nv), kk,
                                                       None if ex is None else int(ex[r]))
            if not (torch.equal(i[r], want_i) and torch.allclose(s[r], want_s, rtol=0, atol=1e-12)):
                bad.append(r)
        return bad

    comm = distributed.GroupComm()
    stats = {}
    s, i = engine.search_shards([shard], Q, k, exclude=excl, comm=comm, n_total=nv, small_nv=1000, stats=stats,
                                label_mask=masks)
    fails = ["rows %s" % b for b in [check(s, i, k, excl)] if b]
    if not (bool((i[3] == -1).all()) and int((i[4] >= 0).sum()) == int((labels == 62).sum()) < k):
        fails.append("padding")
    # (the re-run covers query 1, whose ~3 000 eligible rows all lie near it, and query 7)
    if not (stats.get("reruns", 0) >= 1 and stats["thr_inf_rows"] >= 4):
        fails.append("stats %s" % {x: stats.get(x) for x in ("reruns", "rerun_rows", "thr_inf_rows")})
    if not (stats["eligible_min"] == 0 and stats["eligible_max"] == nv):
        fails.append("eligible %s %s" % (stats["eligible_min"], stats["eligible_max"]))
    # one mask for the whole batch, numpy uint64, and the unfiltered rows of the batch unchanged
    import numpy as np
    s2, i2 = engine.search_shards([shard], Q, k, comm=comm, n_total=nv, small_nv=1000,
                                  label_mask=np.uint64(bit(range(0, 64, 4))))
    m2 = torch.full((nq,), bit(range(0, 64, 4)), dtype=torch.int64)
    exact_m = exact.clone()
    exact_m[~_allowed(m2, labels)] = float("-inf")
    fails += ["one mask: rows %s" % b for b in [check(s2, i2, k)] if b]
    # small-corpus branch across ranks
    exact_m = exact.clone()
    exact_m[~_allowed(masks, labels)] = float("-inf")
    s3, i3 = engine.search_shards([shard], Q, 7, comm=comm, n_total=nv, small_nv=10 ** 9, label_mask=masks)
    fails += ["small: rows %s" % b for b in [check(s3, i3, 7)] if b]
    # relabel rows of rank 0's shard only (every rank makes the same call): both ranks re-reduce the label histogram
    moved = torch.randperm(nv // 2, generator=torch.Generator().manual_seed(12))[:2000]
    shard.set_labels(moved, torch.full((2000,), 62))
    labels[moved] = 62
    exact_m = exact.clone()
    exact_m[~_allowed(masks, labels)] = float("-inf")
    s4, i4 = engine.search_shards([shard], Q, k, exclude=excl, comm=comm, n_total=nv, small_nv=1000,
                                  label_mask=masks)
    fails += ["relabelled: rows %s" % b for b in [check(s4, i4, k, excl)] if b]
    with open(os.path.join(out_dir, "rank%d" % rank), "w") as f:
        f.write("; ".join(fails) if fails else "ok")
    dist.destroy_process_group()


def test_two_rank_filtered_search_on_cpu_model(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        assert open(os.path.join(str(tmp_path), "rank%d" % r)).read() == "ok"
