"""Similar pairs through the multi-rank pipeline on CPU: two gloo ranks, each with a CPU model shard
(tests/cpu_model.py) that also gives suffix views, and torch statements of the selection kernels
(``engine._range_select`` with its ``after`` floor, ``engine._range_merge``).  Covers an uneven split whose blocks
scan rows of both ranks, the all-reduce that brings one rank's stored rows to the other as queries, exact copies held
on different ranks, and a list that overflows the first pass on one rank only -- each against the full-corpus fp64
model.  The kernels themselves are tested on the B200 (test_gpu_similar_pairs.py)."""
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


def _patch_select_kernels(engine):
    def range_select(exact, cand, idx_offset, excl, ms, counts=None, off=None, max_len=0, out_s=None, out_i=None,
                     after=None):
        cnt, _, ci = cand
        rows, cap = ci.shape
        hits = []
        for r in range(rows):
            n = min(int(cnt[r]), cap)
            s, ids = exact[r, :n], ci[r, :n].long() + idx_offset
            keep = (s > -INF) & (s >= ms[r])
            if excl is not None:
                keep &= ids != excl[r]
            if after is not None:
                keep &= ids > after[r]
            hits.append((s[keep], ids[keep]))
        if off is None:
            return torch.tensor([len(h[0]) for h in hits], dtype=torch.int64)
        for r, (s, ids) in enumerate(hits):
            m = int(counts[r])
            if m == 0:
                continue
            assert m == len(s) <= max_len
            s, ids = _order(s, ids)
            out_s[int(off[r]):int(off[r]) + m], out_i[int(off[r]):int(off[r]) + m] = s, ids

    def range_merge(score, idx, seg_off, off, max_len, out_s, out_i):
        for r in range(seg_off.shape[1] - 1):
            runs = [(score[a:b], idx[a:b]) for a, b in zip(seg_off[:, r].tolist(), seg_off[:, r + 1].tolist())]
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

    class Shard(cpu_model.ModelShard):
        def _suffix(self, start):
            start = min(int(start), self.n)
            v = object.__new__(type(self))
            v.__dict__.update(self.__dict__)
            v.raw, v.op = self.raw[start:], self.op[start:]
            v.norm = [x[start:] for x in self.norm]
            v.n, v.index_offset = self.n - start, self.index_offset + start
            v.resid_max2 = self.resid_max2
            return v

    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    cpu_model.patch_engine(setattr)
    _patch_select_kernels(engine)
    engine.PAIR_BLOCK = 256
    engine.RANGE_CAP0 = 64
    nv, dims, wts = 3000, (24, 8), [0.6, 0.4]
    split = 1700                                                # uneven, not a multiple of the block
    g = torch.Generator().manual_seed(5)
    V = torch.randn((nv, sum(dims)), generator=g)
    for j in range(0, nv, 37):                                  # noisy near-copies of earlier rows
        if j:
            src = int(torch.randint(0, j, (1,), generator=g))
            V[j] = V[src] + 0.08 * torch.randn(sum(dims), generator=g)
    V[[100, 1800, 2501]] = V[50].clone()                        # exact copies held on both ranks
    big = torch.arange(300, 1500, 12)                           # 100 exact copies, all on rank 0
    V[big] = V[7].clone()
    lo, hi = (0, split) if rank == 0 else (split, nv)
    shard = Shard(V[lo:hi], dims, index_offset=lo)
    full = Shard(V, dims)
    _, qr, qn, _, _ = full.prepare_queries(V, wts)
    exact = full._exact(qr, qn, wts)                            # [nv, nv] fp64

    fails = []

    def check(res, t, tag):
        off = res.offsets
        if off.numel() != nv + 1:
            fails.append("%s: %d lists" % (tag, off.numel() - 1))
            return
        for i in range(nv):
            s, j = res.scores[off[i]:off[i + 1]], res.idx[off[i]:off[i + 1]]
            want = torch.nonzero(exact[i, i + 1:] >= t).flatten() + i + 1
            ws, wj = _order(exact[i, want], want)
            if not (torch.equal(j, wj) and torch.allclose(s, ws, rtol=0, atol=1e-12)):
                fails.append("%s: row %d (%d vs %d pairs)" % (tag, i, len(j), len(wj)))
                return

    comm = distributed.GroupComm()
    for t in (0.9, 0.55):
        stats = {}
        res = engine.similar_pairs_shards([shard], t, weights=wts, comm=comm, stats=stats)
        check(res, t, "t=%s" % t)
        if stats["blocks"] != 13 or stats["pairs"] != res.idx.numel():
            fails.append("stats %s" % stats)
        if t == 0.9:
            # the copies of row 7 overflow rank 0's first-pass lists only; both ranks re-run them in lockstep
            if not stats["rerun_rows"] > 0:
                fails.append("no re-run")
            i, j, s = res.pairs()
            if not (torch.equal(i, torch.repeat_interleave(torch.arange(nv), res.offsets[1:] - res.offsets[:-1]))
                    and torch.equal(j, res.idx)):
                fails.append("pairs()")
            for a, b in ((50, 100), (50, 1800), (100, 2501), (1800, 2501), (7, 1488)):
                if not bool(((i == a) & (j == b)).any()):
                    fails.append("copy pair %d %d missing" % (a, b))
    res = distributed.sharded_similar_pairs(shard, 0.9, weights=wts)
    check(res, 0.9, "wrapper")
    # one process, the whole corpus
    check(engine.similar_pairs_shards([full], 0.9, weights=wts), 0.9, "solo")
    with open(os.path.join(out_dir, "rank%d" % rank), "w") as f:
        f.write("; ".join(fails) if fails else "ok")
    dist.destroy_process_group()


def test_two_rank_similar_pairs_on_cpu_model(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        assert open(os.path.join(str(tmp_path), "rank%d" % r)).read() == "ok"
