"""Multi-GPU check of the similar-pairs join (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_pairs_sharded.py

Every rank holds one shard of a seeded corpus with planted near-copies and groups of exact copies (one of them larger
than the first-pass lists, so lists are re-run); ``distributed.sharded_similar_pairs`` over NCCL must return, on every
rank, exactly what ONE store holding the whole corpus returns (offsets, rows and fp64 scores identical).  Blocks of
512 rows, so that the shard boundaries fall inside blocks of the schedule's walk and the raw-row all-reduce runs for
every block.
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
    engine.PAIR_BLOCK = 512
    dims, w = (256, 64), (0.7, 0.3)
    nv = 50_001
    V = synth.device_gaussian(nv, sum(dims), 21, dev)                  # same seed on every rank -> same corpus
    g = torch.Generator(device=dev).manual_seed(22)
    src = torch.randint(0, nv, (nv // 40,), generator=g, device=dev)
    dst = torch.randint(0, nv, (nv // 40,), generator=g, device=dev)
    V[dst] = V[src] + 0.2 * torch.randn((len(dst), sum(dims)), generator=g, device=dev)
    V[torch.arange(7, nv, 19, device=dev)[:2500]] = V[3].clone()       # 2 500 exact copies across every shard
    lo, hi = distributed.shard_range(nv, world, rank)
    shard = engine.CorpusStore(hi - lo, dims, device=dev, index_offset=lo).add(V[lo:hi])
    full = engine.CorpusStore(nv, dims, device=dev).add(V)
    ok = True
    for t in (0.95, 0.8):
        ref = full.similar_pairs(t, weights=w)
        stats = {}
        res = distributed.sharded_similar_pairs(shard, t, weights=w, stats=stats)
        same = bool(torch.equal(res.offsets, ref.offsets)) and bool(torch.equal(res.idx, ref.idx)) \
            and bool(torch.equal(res.scores, ref.scores))
        ok = ok and same
        if rank == 0:
            print("nv=%d t=%s: %d pairs, %d re-run rows, %s" % (nv, t, ref.idx.numel(), stats["rerun_rows"],
                                                               "identical" if same else "MISMATCH"), flush=True)
    flag = torch.tensor([0 if ok else 1], device=dev)
    dist.all_reduce(flag)
    if rank == 0:
        print("pairs sharded %s on %d GPUs" % ("ok" if int(flag) == 0 else "MISMATCH", world), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 0 else 1)


if __name__ == "__main__":
    main()
