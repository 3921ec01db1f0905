"""Similar-pairs benchmark on one GPU: every pair of corpus rows with fused score >= 0.9, on a seeded corpus of the C5
shape ((1536 + 512) dims, weights 0.6 / 0.4).

    python tools/pairs_bench.py [--nv 1000000 10000000] [--rounds 2] [--loop-max 1000000] [--out pairs_bench.json]

Corpus (regenerated from the seed on the device, chunk by chunk): Gaussian rows; every 100th row (r % 100 == 99) is
replaced by a noisy copy of an earlier row of its chunk (cosine about 0.95 - 0.98); 16 groups of 64 exact copies of
one vector each are spread over the corpus.  Gaussian rows of 1536 / 512 dims score far below 0.9 with each other, so
the pairs are the planted ones plus whatever the near-copies add by chance.

Per corpus size: the join (``CorpusStore.similar_pairs``) is timed with a host clock around the call ending in a
device synchronise; the FILTER time is summed from CUDA events around every xmve_score_filter launch over the corpus
(``step == 1``); the other phases come from ``stats``.  Effective TFLOP/s counts the algorithmic ``n (n - 1) * 2048``
flop of scoring every unordered pair once (2 flop per multiply-add).  ``verified``: 256 sampled rows' lists against
an fp64 statement over the rows regenerated from the seed (scores within 1e-12 of the minimum may go either way),
and every planted pair found.  Up to ``--loop-max`` rows the same answer is also computed through the range-search
loop (every row a query, 8192 per call, self-matches and mirrored pairs dropped), alternating with the join round
by round, and the two results are compared; larger corpora are timed once.  The device name and power limit are
read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cross_modal_video_engine_b200 import _native as N, engine, synth  # noqa: E402

DIMS, WEIGHTS, T, SEED = (1536, 512), (0.6, 0.4), 0.9, 17
D = sum(DIMS)
CHUNK = 1 << 16
GROUPS, COPIES = 16, 64


def groups(n):
    """Rows of the 16 groups of exact copies: int64 [16, 64]."""
    g = torch.arange(GROUPS)[:, None] * (n // GROUPS) + torch.arange(COPIES)[None, :] * (n // (GROUPS * COPIES)) + 13
    return g


def chunks(n, dev):
    """Yields (first row, fp32 rows [<= CHUNK, D], src, dst) of the corpus: row dst is a noisy copy of row src."""
    gv = synth.device_gaussian(GROUPS, D, SEED + 999_999, dev)
    grp = groups(n).to(dev)
    for c, lo in enumerate(range(0, n, CHUNK)):
        hi = min(n, lo + CHUNK)
        x = synth.device_gaussian(hi - lo, D, SEED * 1_000_003 + c, dev)
        r = torch.arange(lo, hi, device=dev)
        dst = r[r % 100 == 99]
        h = (dst * 2654435761) % 1_000_003
        src = lo + h % (dst - lo)                                   # an earlier row of this chunk
        sigma = 0.2 + 0.13 * (h % 997).double() / 997.0
        g = torch.Generator(device=dev).manual_seed(SEED + 7 * c + 1)
        x[dst - lo] = x[src - lo] + sigma[:, None].float() * torch.randn((len(dst), D), generator=g, device=dev)
        mine = (grp >= lo) & (grp < hi)
        gi = torch.nonzero(mine, as_tuple=True)[0]
        x[grp[mine] - lo] = gv[gi]
        yield lo, x, src, dst


def planted(n, dev):
    """Keys i * n + j (i < j) of the planted pairs: near-copies whose two rows are not group members, and every pair
    inside a group."""
    grp = groups(n).to(dev)
    flat = grp.reshape(-1)
    keys = []
    for lo, x, src, dst in chunks(n, dev):
        ok = ~torch.isin(src, flat) & ~torch.isin(dst, flat) & (src % 100 != 99)
        keys.append(src[ok] * n + dst[ok])
    a, b = torch.triu_indices(COPIES, COPIES, 1, device=dev)
    keys.append((grp[:, a] * n + grp[:, b]).reshape(-1))
    return torch.cat(keys)


def unit(x):
    out, o = [], 0
    for d in DIMS:
        v = x[:, o:o + d].double()
        out.append(v / v.norm(dim=1, keepdim=True))
        o += d
    return out


def verify(n, dev, res, sample=256):
    """256 sampled rows against the fp64 statement, and every planted pair found -> (ok, max abs error)."""
    rows = torch.sort(torch.randperm(n, generator=torch.Generator().manual_seed(5))[:sample]).values.to(dev)
    # the sampled rows themselves, regenerated
    q = torch.empty((sample, D), dtype=torch.float32, device=dev)
    for lo, x, _, _ in chunks(n, dev):
        sel = (rows >= lo) & (rows < lo + x.shape[0])
        q[sel] = x[rows[sel] - lo]
    qn = unit(q)
    hits = []                                                       # (sample, row, score) of scores >= T - 1e-12
    for lo, x, _, _ in chunks(n, dev):
        sc = sum(w * (a @ b.t()) for w, a, b in zip(WEIGHTS, qn, unit(x)))
        si, vj = torch.nonzero(sc >= T - 1e-12, as_tuple=True)
        hits.append((si, vj + lo, sc[si, vj]))
    si, vj, ss = (torch.cat([h[k] for h in hits]) for k in range(3))
    off = res.offsets
    ok, err = True, 0.0
    for s, i in enumerate(rows.tolist()):
        got_i, got_s = res.idx[off[i]:off[i + 1]], res.scores[off[i]:off[i + 1]]
        sel = (si == s) & (vj > i)
        ref_i, ref_s = vj[sel], ss[sel]
        sure = ref_i[ref_s >= T + 1e-12]
        okj = bool(torch.isin(sure, got_i).all()) and bool(torch.isin(got_i, ref_i).all())
        if okj and got_i.numel():
            o = torch.argsort(ref_i)
            pos = torch.searchsorted(ref_i[o], got_i)
            err = max(err, float((ref_s[o][pos] - got_s).abs().max()))
            okj = bool(((got_s[:-1] > got_s[1:]) | ((got_s[:-1] == got_s[1:]) & (got_i[:-1] < got_i[1:]))).all())
        ok = ok and okj
    i, j, _ = res.pairs()
    want = planted(n, dev)
    found = bool(torch.isin(want, i * n + j).all())
    return ok and found and err <= 1e-12, err, found, int(want.numel())


def loop(store, n):
    """The same answer through range_search: every row a query, self-matches and mirrored pairs dropped."""
    counts = torch.zeros((n,), dtype=torch.int64, device=store.device)
    s_parts, i_parts = [], []
    for r0 in range(0, n, engine.PAIR_BLOCK):
        r1 = min(n, r0 + engine.PAIR_BLOCK)
        res = store.range_search(store.raw[r0:r1, :D], T, weights=WEIGHTS)
        row = torch.repeat_interleave(torch.arange(r0, r1, device=store.device), res.offsets[1:] - res.offsets[:-1])
        keep = res.idx > row
        counts[r0:r1] = torch.bincount(row[keep] - r0, minlength=r1 - r0)
        s_parts.append(res.scores[keep])
        i_parts.append(res.idx[keep])
    off = torch.zeros((n + 1,), dtype=torch.int64, device=store.device)
    off[1:] = torch.cumsum(counts, 0)
    return engine.RangeResult(off, torch.cat(s_parts), torch.cat(i_parts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nv", type=int, nargs="+", default=[1_000_000])
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--loop-max", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    filt = []
    call0 = N.call

    def call(name, *a):
        if name == "xmve_score_filter" and a[6] == 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = call0(name, *a)
            e1.record()
            filt.append((e0, e1))
            return r
        return call0(name, *a)

    def timed(fn):
        filt.clear()
        N.call = call
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3
        N.call = call0
        return out, ms, sum(a.elapsed_time(b) for a, b in filt)

    cases = {}
    for n in args.nv:
        store = engine.CorpusStore(n, DIMS, device=dev)
        for _, x, _, _ in chunks(n, dev):
            store.add(x)
        flop = n * (n - 1) * D                                      # n (n - 1) / 2 pairs x 2 D flop
        fns = {"join": lambda: store.similar_pairs(T, weights=WEIGHTS)}
        if n <= args.loop_max:
            fns["range_search_loop"] = lambda: loop(store, n)
        # warm-up: a join over the first 64 k rows (every kernel shape the blocks use)
        engine.similar_pairs_shards([store._suffix(n - min(n, 1 << 16))], T, weights=WEIGHTS)
        rounds = args.rounds if n <= args.loop_max else 1
        r = {x: {"ms": [], "filter_ms": []} for x in fns}
        outs = {}
        for _ in range(rounds):
            for x, fn in fns.items():
                outs[x], ms, f = timed(fn)
                r[x]["ms"].append(ms)
                r[x]["filter_ms"].append(f)
        for x in fns:
            best = min(range(rounds), key=lambda k: r[x]["ms"][k])
            r[x]["ms_best"], r[x]["filter_ms_of_best"] = r[x]["ms"][best], r[x]["filter_ms"][best]
            r[x]["effective_tflops"] = flop / (r[x]["ms_best"] * 1e-3) / 1e12
        st = {}
        res = store.similar_pairs(T, weights=WEIGHTS, stats=st)
        r["join"].update({"eps": st["eps"], "blocks": st["blocks"], "candidates": st["candidates"],
                          "pairs": st["pairs"], "rerun_rows": st["rerun_rows"], "passes": st["passes"],
                          "phases_ms": st["phases_ms"],
                          "filter_tflops": flop / (r["join"]["filter_ms_of_best"] * 1e-3) / 1e12})
        if "range_search_loop" in outs:
            lp = outs["range_search_loop"]
            r["loop_equals_join"] = bool(torch.equal(lp.offsets, res.offsets) and torch.equal(lp.idx, res.idx)
                                         and torch.equal(lp.scores, res.scores))
            r["join_over_loop"] = r["join"]["ms_best"] / r["range_search_loop"]["ms_best"]
        del outs
        ok, err, found, n_planted = verify(n, dev, res)
        r.update({"verified": ok, "verify_max_abs_err": err, "planted_pairs": n_planted, "planted_all_found": found})
        cases["nv_%d" % n] = r
        print(n, json.dumps(r), flush=True)
        del store, res
        torch.cuda.empty_cache()
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        smi = "unavailable"
    doc = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": smi, "dims": list(DIMS),
           "weights": list(WEIGHTS), "min_score": T, "pair_block": engine.PAIR_BLOCK, "rounds": args.rounds,
           "cases": cases}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
