"""Multi-GPU check of the filtered search (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_filtered_sharded.py

Every rank holds one shard of a seeded, labelled corpus; ``distributed.sharded_search(..., label_mask=...)`` over NCCL
must return, on every rank, exactly what ONE store holding the whole corpus returns (indices and fp64 scores
identical): per-query masks from every label down to none, with and without exclusions, for the filtered path and the
small-corpus path, and again after ``set_labels`` -- a collective call, every rank passes the same global ids --
first of rows spread over all shards, then of rows of rank 0's shard only.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cross_modal_video_engine_b200 import distributed, engine, synth  # noqa: E402


def _masks(nq, g):
    """All labels, ~30 %, ~5 %, one rare label, none, then random 16-label masks."""
    def bits(ls):
        m = sum(1 << int(x) for x in ls)
        return m - (1 << 64) if m >= (1 << 63) else m
    base = [-1, bits(range(19)), bits(range(3)), bits([63]), 0]
    return torch.tensor([base[q] if q < len(base) else bits(torch.randperm(64, generator=g)[:16]) for q in range(nq)],
                        dtype=torch.int64)


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    dims, w = (256, 64), (0.7, 0.3)
    ok = True
    for nv, nq, k in ((600_000, 300, 100), (9_000, 64, 10), (300_001, 7, 1000)):
        V = synth.device_gaussian(nv, sum(dims), 11, dev)             # same seed on every rank -> same corpus
        Q = synth.device_gaussian(nq, sum(dims), 12, dev)
        g = torch.Generator().manual_seed(nv)
        labels = torch.randint(0, 63, (nv,), generator=g)
        labels[torch.randperm(nv, generator=g)[:50]] = 63              # a label with fewer rows than k
        masks = _masks(nq, g)
        lo, hi = distributed.shard_range(nv, world, rank)
        shard = engine.CorpusStore(hi - lo, dims, device=dev, index_offset=lo).add(V[lo:hi], labels=labels[lo:hi])
        full = engine.CorpusStore(nv, dims, device=dev).add(V, labels=labels)
        excl = torch.randint(0, nv, (nq,), generator=torch.Generator().manual_seed(5)).numpy()
        lo0, hi0 = distributed.shard_range(nv, world, 0)
        relabel = {"relabelled": torch.randperm(nv, generator=g)[:nv // 10],
                   "rank-0 rows relabelled": lo0 + torch.randperm(hi0 - lo0, generator=g)[:(hi0 - lo0) // 10]}
        for state in ("added", "relabelled", "rank-0 rows relabelled"):
            if state != "added":
                ids = relabel[state]
                new = torch.randint(0, 64, (len(ids),), generator=g)
                full.set_labels(ids, new)
                shard.set_labels(ids, new)
            for ex in (None, excl):
                s_ref, i_ref = full.search(Q, k, weights=w, exclude=ex, label_mask=masks)
                s, i = distributed.sharded_search(shard, Q, k, weights=w, exclude=ex, n_total=nv, label_mask=masks)
                same = bool(torch.equal(i, i_ref)) and bool(torch.equal(s, s_ref))
                ok = ok and same
                if rank == 0:
                    print("nv=%d nq=%d k=%d %s exclude=%s: %s" % (nv, nq, k, state, ex is not None,
                                                                   "identical" if same else "MISMATCH"), flush=True)
        del shard, full, V
        torch.cuda.empty_cache()
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    if rank == 0:
        print("filtered sharded search on %d GPUs: %s" % (world, "OK" if int(flag) == 0 else "MISMATCH"), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 0 else 1)


if __name__ == "__main__":
    main()
