"""Range search and range count through the multi-rank pipeline on CPU: two gloo ranks, each with a CPU model shard
(tests/cpu_model.py) and torch statements of the two range kernels (``engine._range_select`` / ``_range_merge``).
Covers the all-gathered list sizes and the overflow re-run in lockstep when only one rank's list overflows, the
gathered counts, the padded packed blocks and the merge, ``range_count``'s all-reduce, and the exclusion of a row
that the other rank owns -- each against the full-corpus fp64 model.  The kernels themselves are tested on the B200
(test_gpu_range_search.py)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT

INF = float("inf")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _order(s, i):
    """(score desc, row asc) order of the pairs (s, i)."""
    o = torch.argsort(i, stable=True)
    s, i = s[o], i[o]
    o = torch.argsort(s, descending=True, stable=True)
    return s[o], i[o]


def _patch_range_kernels(engine):
    def range_select(exact, cand, idx_offset, excl, ms, counts=None, off=None, max_len=0, out_s=None, out_i=None):
        cnt, _, ci = cand
        rows, cap = ci.shape
        hits = []
        for r in range(rows):
            n = min(int(cnt[r]), cap)
            s, ids = exact[r, :n], ci[r, :n].long() + idx_offset
            keep = (s > -INF) & (s >= ms[r])
            if excl is not None:
                keep &= ids != excl[r]
            hits.append((s[keep], ids[keep]))
        if off is None:
            return torch.tensor([len(h[0]) for h in hits], dtype=torch.int64)
        for r, (s, ids) in enumerate(hits):
            m = int(counts[r])
            if m == 0:                                              # (a row a later pass owns)
                continue
            assert m == len(s) <= max_len
            s, ids = _order(s, ids)
            out_s[int(off[r]):int(off[r]) + m], out_i[int(off[r]):int(off[r]) + m] = s, ids

    def range_merge(score, idx, seg_off, off, max_len, out_s, out_i):
        for r in range(seg_off.shape[1] - 1):
            runs = [(score[a:b], idx[a:b]) for a, b in zip(seg_off[:, r].tolist(), seg_off[:, r + 1].tolist())]
            for s, i in runs:                                       # every shard's run arrives sorted
                assert torch.equal(_order(s, i)[1], i)
            s, i = _order(torch.cat([x[0] for x in runs]), torch.cat([x[1] for x in runs]))
            assert len(s) == int(off[r + 1] - off[r]) <= max_len
            out_s[int(off[r]):int(off[r + 1])], out_i[int(off[r]):int(off[r + 1])] = s, i

    engine._range_select = range_select
    engine._range_merge = range_merge


def _worker(rank, world, port, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from cross_modal_video_engine_b200 import distributed, engine
    import cpu_model
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cpu_model.patch_engine(setattr)
    _patch_range_kernels(engine)
    nv, nq, d = 40000, 10, 32
    g = torch.Generator().manual_seed(21)
    V, Q = torch.randn((nv, d), generator=g), torch.randn((nq, d), generator=g)
    for qi in range(nq):                                        # planted neighbours
        rows = torch.randperm(nv, generator=g)[:30]
        V[rows] = Q[qi] + 0.3 * torch.randn((30, d), generator=g)
    dense = torch.randperm(nv // 2, generator=g)[:3500]         # query 2: 3 500 close rows, all on rank 0
    V[dense] = Q[2] * 2.0 + 0.4 * torch.randn((len(dense), d), generator=g)
    lo, hi = distributed.shard_range(nv, world, rank)
    shard = cpu_model.ModelShard(V[lo:hi], (d,), index_offset=lo)
    full = cpu_model.ModelShard(V, (d,))
    _, qr, qn, _, _ = full.prepare_queries(Q, [1.0])
    exact = full._exact(qr, qn, [1.0])                          # [nq, nv] fp64

    def between(q, j):
        """a minimum midway between the j-th and (j+1)-th best exact scores of query q"""
        top = torch.sort(exact[q], descending=True).values
        return float(0.5 * (top[j - 1] + top[j]))

    ms = torch.tensor([between(q, j) for q, j in enumerate((5, 40, 3000, 1, 12, 100, 7, 25, 30, 2))],
                      dtype=torch.float64)
    ms[6], ms[7] = INF, -INF                                    # an empty list and the whole corpus
    excl = torch.full((nq,), -1, dtype=torch.int64)
    for q, owner in ((0, 1), (5, 0)):                           # exclude in-range rows: each rank owns one
        o_lo, o_hi = distributed.shard_range(nv, world, owner)
        inside = torch.nonzero(exact[q] >= ms[q]).flatten()
        excl[q] = int(inside[(inside >= o_lo) & (inside < o_hi)][0])
    excl[7] = 3                                                 # (-inf: every row but one of rank 0's)

    def want(q, m, ex=None):
        ids = torch.nonzero(exact[q] >= m).flatten()
        if ex is not None and int(ex[q]) >= 0:
            ids = ids[ids != int(ex[q])]
        return _order(exact[q, ids], ids)

    fails = []

    def check(res, mins, ex, tag):
        off = res.offsets
        for q in range(nq):
            s, i = res.scores[off[q]:off[q + 1]], res.idx[off[q]:off[q + 1]]
            ws, wi = want(q, float(mins[q]), ex)
            if not (torch.equal(i, wi) and torch.allclose(s, ws, rtol=0, atol=1e-12)):
                fails.append("%s: query %d (%d vs %d rows)" % (tag, q, len(i), len(wi)))

    comm = distributed.GroupComm()
    stats = {}
    res = engine.range_search_shards([shard], Q, ms, exclude=excl, comm=comm, stats=stats)
    check(res, ms, excl, "per-query")
    # rank 0's list of query 2 and both ranks' lists of query 7 overflow the first pass; both ranks re-run them
    if not (stats["passes"] == 1 and stats["rerun_rows"] == 2):
        fails.append("re-run %s %s" % (stats["passes"], stats["rerun_rows"]))
    cnt = engine.range_count_shards([shard], Q, ms, exclude=excl, comm=comm)
    if not torch.equal(cnt, res.offsets[1:] - res.offsets[:-1]):
        fails.append("range_count %s vs %s" % (cnt.tolist(), (res.offsets[1:] - res.offsets[:-1]).tolist()))
    # a scalar minimum, no exclusions, through the distributed wrappers
    r0 = float(ms[1])
    res2 = distributed.sharded_range_search(shard, Q, r0)
    check(res2, [r0] * nq, None, "scalar")
    cnt2 = distributed.sharded_range_count(shard, Q, r0)
    if not torch.equal(cnt2, torch.tensor([int((exact[q] >= r0).sum()) for q in range(nq)])):
        fails.append("scalar range_count")
    # padded(): the CSR as [nq, max_count] rows, -inf / -1 padded
    ps, pi = res.padded()
    lens = (res.offsets[1:] - res.offsets[:-1]).tolist()
    if not (pi.shape[1] == max(lens) and all(int((pi[q] >= 0).sum()) == lens[q] for q in range(nq))
            and bool((ps[6] == -INF).all())):
        fails.append("padded")
    with open(os.path.join(out_dir, "rank%d" % rank), "w") as f:
        f.write("; ".join(fails) if fails else "ok")
    dist.destroy_process_group()


def test_two_rank_range_search_on_cpu_model(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        assert open(os.path.join(str(tmp_path), "rank%d" % r)).read() == "ok"
