"""Range-search benchmark on one GPU: the C5-shaped corpus of bench.py (10 M x (1536 + 512), weights 0.6 / 0.4) and
8192 queries.

    python tools/range_bench.py [--nv 10000000] [--nq 8192] [--steps 2] [--rounds 3] [--out range_bench.json]

Cases:
- ``matched_k{10,100,1000}``: per-query ``min_score`` = the k-th score ``search(q, k)`` returns.  Range search and the
  top-k search at the same depth alternate round by round; both are timed (host clock around ``steps`` calls ending
  in a device synchronise).  Every range list must start with the top-k list (``topk_prefix_ok``).
- ``scalar_100``: one ``min_score`` for all queries, the median over queries of the 100th score, i.e. about 100
  results per query on average, more for queries in dense regions (a list longer than the first pass's 2048
  entries is re-run).
- ``range_count`` at every one of these thresholds, timed alternating with the range search.

Per case: ms per call, FILTER ms per call (CUDA events around every full-corpus xmve_score_filter /
xmve_score_filter_labeled launch), candidates and results per query, re-run rows and passes, the phase times of
``stats`` (median of three calls), and ``verified``: 128 queries against an fp64 statement over corpus rows
regenerated from the seed (rows within 1e-12 of the minimum may go either way).  The device name and power limit
are read in the same process.
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
import bench  # noqa: E402  (C5 corpus generator and constants)
from cross_modal_video_engine_b200 import _native as N, engine, synth  # noqa: E402


def fp64_scores(chunks, q_sub):
    """Yields (first row, fp64 scores [len(q_sub), rows]) over the regenerated corpus."""
    offs = [0]
    for d in bench.DIMS:
        offs.append(offs[-1] + d)
    qn = [q_sub[:, a:b].double() / q_sub[:, a:b].double().norm(dim=1, keepdim=True) for a, b in zip(offs, offs[1:])]
    for lo, rows in chunks:
        sc = torch.zeros((q_sub.shape[0], rows.shape[0]), dtype=torch.float64, device=q_sub.device)
        for w, q, (a, b) in zip(bench.WEIGHTS, qn, zip(offs, offs[1:])):
            v = rows[:, a:b].double()
            v /= v.norm(dim=1, keepdim=True)
            sc.addmm_(q, v.t(), alpha=w)
        yield lo, sc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nv", type=int, default=bench.NV_TOTAL)
    ap.add_argument("--nq", type=int, default=bench.NQ)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    store = engine.CorpusStore(args.nv, bench.DIMS, device=dev)
    for _, rows in bench.c5_chunks(synth, torch, dev, 0, args.nv):
        store.add(rows)
    q = synth.device_gaussian(args.nq, sum(bench.DIMS), bench.SEED + 1, dev)
    w = bench.WEIGHTS

    filt = []                                                # (start, end) events of the full-corpus FILTER passes
    call0 = N.call

    def call(name, *a):
        if name in ("xmve_score_filter", "xmve_score_filter_labeled") and a[6] == 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = call0(name, *a)
            e1.record()
            filt.append((e0, e1))
            return r
        return call0(name, *a)

    def timed(fn):
        """ms per call and FILTER ms per call over ``steps`` calls."""
        filt.clear()
        N.call = call
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / args.steps
        N.call = call0
        return ms, sum(a.elapsed_time(b) for a, b in filt) / args.steps

    def med(xs):
        return sorted(xs)[len(xs) // 2]

    cases, tops = {}, {}
    for k in (10, 100, 1000):
        s, i = store.search(q, k, weights=w)
        tops[k] = (s, i)
        cases["matched_k%d" % k] = s[:, k - 1].contiguous()
    cases["scalar_100"] = torch.full((args.nq,), float(tops[100][0][:, 99].median()), dtype=torch.float64, device=dev)

    res = {}
    for name, ms in cases.items():
        k = int(name.split("_k")[1]) if name.startswith("matched") else None
        fns = {"range_search": lambda: store.range_search(q, ms, weights=w),
               "range_count": lambda: store.range_count(q, ms, weights=w)}
        if k is not None:
            fns["search"] = lambda: store.search(q, k, weights=w)
        for fn in fns.values():                              # warm-up of every shape
            fn()
        r = {x: {"ms_per_call": [], "filter_ms_per_call": []} for x in fns}
        for _ in range(args.rounds):
            for x, fn in fns.items():
                t, f = timed(fn)
                r[x]["ms_per_call"].append(t)
                r[x]["filter_ms_per_call"].append(f)
        for x in fns:
            r[x]["ms_per_call_median"] = med(r[x]["ms_per_call"])
            r[x]["filter_ms_per_call_median"] = med(r[x]["filter_ms_per_call"])
        phases = []
        for _ in range(3):                                   # phase times: the median of three calls, phase by phase
            st = {}
            out = store.range_search(q, ms, weights=w, stats=st)
            phases.append(st["phases_ms"])
        st["phases_ms"] = {x: med([p[x] for p in phases]) for x in phases[0]}
        cnt = store.range_count(q, ms, weights=w)
        lens = out.offsets[1:] - out.offsets[:-1]
        r["range_search"].update({"eps": st["eps"], "candidates_per_query": st["candidates_per_query"],
                                  "results_per_query": st["results_per_query"], "results_max": int(lens.max()),
                                  "rerun_rows": st["rerun_rows"], "passes": st["passes"], "phases_ms": st["phases_ms"]})
        r["range_count_equals_lengths"] = bool(torch.equal(cnt, lens))
        if k is not None:
            s, i = tops[k]
            off = out.offsets.cpu()
            r["topk_prefix_ok"] = all(torch.equal(out.idx[off[j]:off[j] + k], i[j]) for j in range(args.nq))
        r["_out"] = out
        res[name] = r
        print(name, {x: r[x]["ms_per_call_median"] for x in fns}, "results/query %.1f" % st["results_per_query"],
              "rerun rows", st["rerun_rows"], flush=True)

    # verification: 128 queries against the fp64 statement, one regeneration of the corpus for every case
    sub = torch.arange(0, args.nq, max(1, args.nq // 128), device=dev)[:128]
    mins = {name: cases[name][sub] for name in cases}
    hits = {name: [] for name in cases}                    # (query, row, score) of rows >= min - 1e-12
    for lo, sc in fp64_scores(bench.c5_chunks(synth, torch, dev, 0, args.nv), q[sub]):
        for name, m in mins.items():
            qq, vv = torch.nonzero(sc >= (m - 1e-12)[:, None], as_tuple=True)
            hits[name].append((qq, vv + lo, sc[qq, vv]))
    for name, r in res.items():
        out = r.pop("_out")
        qq = torch.cat([h[0] for h in hits[name]])
        vv = torch.cat([h[1] for h in hits[name]])
        ss = torch.cat([h[2] for h in hits[name]])
        ok, err = True, 0.0
        off = out.offsets.cpu()
        for j, qi in enumerate(sub.tolist()):
            got_i, got_s = out.idx[off[qi]:off[qi + 1]], out.scores[off[qi]:off[qi + 1]]
            sel = qq == j
            ref_i, ref_s = vv[sel], ss[sel]
            sure = ref_i[ref_s >= mins[name][j] + 1e-12]
            okj = bool(torch.isin(sure, got_i).all()) and bool(torch.isin(got_i, ref_i).all())
            if okj and got_i.numel():
                o = torch.argsort(ref_i)
                pos = torch.searchsorted(ref_i[o], got_i)
                err = max(err, float((ref_s[o][pos] - got_s).abs().max()))
                srt = bool(((got_s[:-1] > got_s[1:]) | ((got_s[:-1] == got_s[1:]) & (got_i[:-1] < got_i[1:]))).all())
                okj = okj and srt
            ok = ok and okj
        r["verify_max_abs_err"] = err
        r["verified"] = ok and err <= 1e-12
        print(name, "verified", r["verified"], flush=True)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        smi = "unavailable"
    doc = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": smi, "nv": args.nv,
           "nq": args.nq, "dims": list(bench.DIMS), "weights": list(w), "steps": args.steps, "rounds": args.rounds,
           "cases": res}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
