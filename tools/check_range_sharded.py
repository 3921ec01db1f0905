"""Multi-GPU check of the range search (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_range_sharded.py

Every rank holds one shard of a seeded corpus; ``distributed.sharded_range_search`` / ``sharded_range_count`` over
NCCL must return, on every rank, exactly what ONE store holding the whole corpus returns (offsets, rows and fp64 scores
identical): per-query minima from a handful of rows to tens of thousands (the re-run of overflowed lists), +inf and
-inf on the small corpus, with and without exclusions and label masks.
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cross_modal_video_engine_b200 import distributed, engine, synth  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    dims, w = (256, 64), (0.7, 0.3)
    ok = True
    for nv, nq, depths in ((600_000, 300, (5, 200, 3000, 30000)), (9_000, 64, (1, 50, 9000, 0))):
        V = synth.device_gaussian(nv, sum(dims), 11, dev)             # same seed on every rank -> same corpus
        Q = synth.device_gaussian(nq, sum(dims), 12, dev)
        g = torch.Generator().manual_seed(nv)
        labels = torch.randint(0, 64, (nv,), generator=g)
        lo, hi = distributed.shard_range(nv, world, rank)
        shard = engine.CorpusStore(hi - lo, dims, device=dev, index_offset=lo).add(V[lo:hi], labels=labels[lo:hi])
        full = engine.CorpusStore(nv, dims, device=dev).add(V, labels=labels)
        # minima at the given depths: +inf for depth 0, -inf beyond the corpus, else bisected with the full store's
        # range_count until at least d and at most 1.05 d + 5 rows reach them
        want = torch.tensor([depths[q % len(depths)] for q in range(nq)], dtype=torch.float64)
        lo_s, hi_s = torch.full((nq,), -1.0, dtype=torch.float64), torch.full((nq,), 1.0, dtype=torch.float64)
        for _ in range(40):
            mid = 0.5 * (lo_s + hi_s)
            c = full.range_count(Q, mid, weights=w).cpu().double()
            lo_s = torch.where(c > 1.05 * want + 5, mid, lo_s)
            hi_s = torch.where(c < want, mid, hi_s)
        ms = torch.where(want == 0, float("inf"), torch.where(want >= nv, float("-inf"), 0.5 * (lo_s + hi_s)))
        excl = torch.randint(0, nv, (nq,), generator=torch.Generator().manual_seed(5))
        masks = torch.randint(-(1 << 62), 1 << 62, (nq,), generator=g)
        for ex, lm in ((None, None), (excl, None), (excl, masks)):
            ref = full.range_search(Q, ms, weights=w, exclude=ex, label_mask=lm)
            res = distributed.sharded_range_search(shard, Q, ms, weights=w, exclude=ex, label_mask=lm)
            cnt = distributed.sharded_range_count(shard, Q, ms, weights=w, exclude=ex, label_mask=lm)
            same = bool(torch.equal(res.offsets, ref.offsets)) and bool(torch.equal(res.idx, ref.idx)) \
                and bool(torch.equal(res.scores, ref.scores)) and bool(torch.equal(cnt, ref.offsets[1:] - ref.offsets[:-1]))
            ok = ok and same
            if rank == 0:
                print("nv=%d nq=%d exclude=%s mask=%s: %d results, %s" % (
                    nv, nq, ex is not None, lm is not None, ref.idx.numel(), "identical" if same else "MISMATCH"),
                    flush=True)
        del shard, full, V
        torch.cuda.empty_cache()
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    if rank == 0:
        print("range sharded %s on %d GPUs" % ("ok" if int(flag) == 0 else "MISMATCH", world), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 0 else 1)


if __name__ == "__main__":
    main()
