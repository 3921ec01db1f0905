"""Filtered-search benchmark on one GPU: the C5-shaped corpus of bench.py (10 M x (1536 + 512), 8192 queries, top-100)
with labels uniform over 64 values, searched with masks that select 64, 16, 4 and 1 labels (100 %, 25 %, 6.25 %,
1.56 % of the rows) and without a mask, the five alternating round by round.  A second phase relabels the corpus so
that label 63 holds only ``--rare`` rows (few enough for the candidate lists: those queries get thr = -inf and the
FILTER lists every eligible row) and alternates the unfiltered search, a mask selecting that rare label, and a mask
of 0 (no eligible row: thr = +inf).

    python tools/filter_bench.py [--nv 10000000] [--nq 8192] [--steps 5] [--rounds 3] [--out filter_bench.json]

Per configuration: ms per search step (host clock around ``steps`` searches ending in a device synchronise), the
FILTER pass over the whole corpus in ms (CUDA events around the xmve_score_filter / xmve_score_filter_labeled launch
with b_row_step == 1), candidates and rescored rows per query, rows re-run, and ``verified``: 128 queries checked
against an fp64 statement over corpus rows regenerated from the seed (ineligible rows excluded).  The device name and
power limit are read in the same process.
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

LABEL_SEED = 77


def _mask(n_labels):
    m = (1 << n_labels) - 1
    return m - (1 << 64) if m >= (1 << 63) else m


def _labels(nv, device):
    g = torch.Generator(device=device).manual_seed(LABEL_SEED)
    return torch.randint(0, 64, (nv,), generator=g, device=device, dtype=torch.int64)


def fp64_topk_masked(chunks, q_sub, labels, mask, k):
    """bench.fp64_topk_regenerated restricted to the rows whose label bit is set in ``mask`` (one mask for all)."""
    def masked():
        for lo, rows in chunks:
            m = torch.tensor(mask, dtype=torch.int64, device=labels.device)
            ok = torch.bitwise_and(torch.bitwise_right_shift(m, labels[lo:lo + rows.shape[0]]), 1) != 0
            yield lo, rows, ok
    offs = [0]
    for d in bench.DIMS:
        offs.append(offs[-1] + d)
    qn = [q_sub[:, a:b].double() / q_sub[:, a:b].double().norm(dim=1, keepdim=True) for a, b in zip(offs, offs[1:])]
    best_s = torch.empty((q_sub.shape[0], 0), dtype=torch.float64, device=q_sub.device)
    best_i = torch.empty((q_sub.shape[0], 0), dtype=torch.int64, device=q_sub.device)
    for lo, rows, ok in masked():
        sc = torch.zeros((q_sub.shape[0], rows.shape[0]), dtype=torch.float64, device=q_sub.device)
        for w, q, (a, b) in zip(bench.WEIGHTS, qn, zip(offs, offs[1:])):
            v = rows[:, a:b].double()
            v /= v.norm(dim=1, keepdim=True)
            sc.addmm_(q, v.t(), alpha=w)
        sc[:, ~ok] = float("-inf")
        top_s, top_i = torch.topk(sc, min(k, rows.shape[0]), dim=1)
        best_s, best_i = torch.cat([best_s, top_s], 1), torch.cat([best_i, top_i + lo], 1)
        o = torch.argsort(best_s, dim=1, descending=True, stable=True)[:, :4 * k]
        best_s, best_i = torch.gather(best_s, 1, o), torch.gather(best_i, 1, o)
    o = torch.argsort(best_i, dim=1, stable=True)
    best_s, best_i = torch.gather(best_s, 1, o), torch.gather(best_i, 1, o)
    o = torch.argsort(best_s, dim=1, descending=True, stable=True)[:, :k]
    s, i = torch.gather(best_s, 1, o), torch.gather(best_i, 1, o)
    return s, torch.where(s > float("-inf"), i, torch.full_like(i, -1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nv", type=int, default=bench.NV_TOTAL)
    ap.add_argument("--nq", type=int, default=bench.NQ)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--rare", type=int, default=10_000, help="rows left with label 63 in the second phase")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    k = bench.TOPK
    store = engine.CorpusStore(args.nv, bench.DIMS, device=dev)
    labels = _labels(args.nv, dev)
    for lo, rows in bench.c5_chunks(synth, torch, dev, 0, args.nv):
        store.add(rows, labels=labels[lo:lo + rows.shape[0]])
    q = synth.device_gaussian(args.nq, sum(bench.DIMS), bench.SEED + 1, dev)
    configs = [("unfiltered", None), ("64_labels", _mask(64)), ("16_labels", _mask(16)), ("4_labels", _mask(4)),
               ("1_label", _mask(1))]

    filt = []                                                # (start, end) events of the full-corpus FILTER
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

    def search(m):
        return store.search(q, k, weights=bench.WEIGHTS, label_mask=m)

    sub = torch.arange(0, args.nq, max(1, args.nq // 128), device=dev)[:128]

    def measure(configs, res):
        for _, m in configs:                                 # warm-up of every shape
            search(m)
        torch.cuda.synchronize()
        for name, _ in configs:
            res[name] = {"ms_per_step": [], "filter_ms": []}
        N.call = call
        for _ in range(args.rounds):
            for name, m in configs:
                filt.clear()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    search(m)
                torch.cuda.synchronize()
                res[name]["ms_per_step"].append((time.perf_counter() - t0) * 1e3 / args.steps)
                res[name]["filter_ms"].append(sum(a.elapsed_time(b) for a, b in filt) / max(len(filt), 1))
        N.call = call0
        for name, m in configs:
            r = res[name]
            st = {}
            s, i = store.search(q, k, weights=bench.WEIGHTS, label_mask=m, stats=st)
            r["ms_per_step_median"] = sorted(r["ms_per_step"])[len(r["ms_per_step"]) // 2]
            r["filter_ms_median"] = sorted(r["filter_ms"])[len(r["filter_ms"]) // 2]
            r["candidates_per_query"] = float(sum(c.float().mean() for c in st["cand_count"]))
            r["rescored_per_query"] = st["rescored_per_query"]
            r["rerun_rows"] = st.get("rerun_rows", 0)
            if m is not None:
                r["eligible_min"], r["eligible_max"] = st["eligible_min"], st["eligible_max"]
                r["thr_inf_rows"] = st["thr_inf_rows"]
            ref_s, ref_i = fp64_topk_masked(bench.c5_chunks(synth, torch, dev, 0, args.nv), q[sub], labels,
                                            -1 if m is None else m, k)
            err = float((ref_s - s[sub]).abs().nan_to_num(0.0).max())
            r["verify_max_abs_err"] = err
            r["verified"] = bool(torch.equal(ref_i, i[sub])) and err <= 1e-12
            print(name, {x: r[x] for x in ("ms_per_step_median", "filter_ms_median", "candidates_per_query",
                                            "rescored_per_query", "rerun_rows", "verified")}, flush=True)
        base = res[configs[0][0]]["filter_ms_median"]
        for name, _ in configs:
            res[name]["filter_vs_unfiltered"] = res[name]["filter_ms_median"] / base

    res = {}
    measure(configs, res)
    # phase 2: label 63 keeps `rare` rows, the others move to label 62
    ids = torch.nonzero(labels == 63).flatten()[args.rare:]
    labels[ids] = 62
    store.set_labels(ids, labels[ids])
    res2 = {}
    measure([("unfiltered", None), ("rare_label", -(1 << 63)), ("mask_0", 0)], res2)
    res["unfiltered_after_relabel"] = res2.pop("unfiltered")      # the reference of the two below
    res.update(res2)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        smi = "unavailable"
    out = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": smi, "nv": args.nv,
           "nq": args.nq, "k": k, "dims": list(bench.DIMS), "steps": args.steps, "rounds": args.rounds, "rare": args.rare,
           "configs": res}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
