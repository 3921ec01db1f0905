"""Search on small corpora (at most 16 384 rows) on one GPU: the certified filter pipeline of ``search_shards``
against the former fp64-matrix path, which formed the whole ``[nq, n]`` fp64 score matrix with the DMMA kernel
and selected from it without a certificate.  The former path is restated here from the same kernels, so that both
alternate within one process.

    python tools/small_bench.py [--rounds 7] [--steps 20] [--out small_bench.json]

Shapes:
- ``c1``: 1 000 queries x 1 000 rows x 1 536 dims, k = 10 (C1, the AVS-style corpus);
- ``mf``: 4 096 queries x 2 300 rows x 640 dims, ``norm_mode="eps"``, k = 50 (a MultiFusion-sized index).

Per shape: ms per call for the former path (eager), ``search`` (eager) and a captured ``GraphSearch`` replay; each
figure is the median over ``rounds`` rounds of ``steps`` calls (host clock, ending in a device synchronise), the
three alternating round by round.  ``same_idx`` says whether ``search`` returned the former path's indices, and
``max_abs_score_diff`` how far its scores are from the former path's.  The device name and power limit are read in
the same process.
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

SHAPES = {"c1": dict(nq=1000, nv=1000, d=1536, k=10, norm="plain"),
          "mf": dict(nq=4096, nv=2300, d=640, k=50, norm="eps")}


def fp64_matrix_search(store, q, k):
    """The former path for one single-space store: K1 on the queries, both sides normalised in fp64, the DMMA fp64
    score matrix, the bitonic top-k without a certificate."""
    st = N.stream_ptr()
    _, q_raw, _, _, nq = store.prepare_queries(q)
    d, n = store.dims[0], store.n
    qn = torch.empty((nq, d), dtype=torch.float64, device=store.device)
    vn = torch.empty((n, d), dtype=torch.float64, device=store.device)
    N.call("xmve_normalize_f64", N.ptr(q_raw), N.F32, nq, d, q_raw.stride(0), N.ptr(qn), d, store.norm_mode, st)
    N.call("xmve_normalize_f64", N.ptr(store.raw), N.F32, n, d, store.raw.stride(0), N.ptr(vn), d, store.norm_mode, st)
    sc = torch.empty((nq, n), dtype=torch.float64, device=store.device)
    N.call("xmve_score_f64", N.ptr(qn), nq, d, N.ptr(vn), n, d, d, 1.0, N.ptr(sc), n, st)
    s_ = torch.empty((nq, k), dtype=torch.float64, device=store.device)
    i_ = torch.empty((nq, k), dtype=torch.int64, device=store.device)
    N.call("xmve_select_topk_i32", N.ptr(sc), None, nq, n, None, store.index_offset, None, k, None, 0.0, None, None,
           N.ptr(s_), N.ptr(i_), None, None, None, None, st)
    return s_, i_


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 / args.steps

    res = {}
    for name, sh in SHAPES.items():
        V = torch.from_numpy(synth.gaussian(11, sh["nv"], sh["d"]))
        q = torch.from_numpy(synth.gaussian(12, sh["nq"], sh["d"])).to(dev)
        store = engine.CorpusStore(sh["nv"], (sh["d"],), device=dev, norm_mode=sh["norm"]).add(V)
        k = sh["k"]
        gs = engine.GraphSearch(store, sh["nq"], k)
        fns = {"fp64_matrix_eager": lambda: fp64_matrix_search(store, q, k),
               "search_eager": lambda: store.search(q, k),
               "graph_replay": lambda: gs(q)}
        outs = {x: fn() for x, fn in fns.items()}            # warm-up of every shape
        times = {x: [] for x in fns}
        for _ in range(args.rounds):
            for x, fn in fns.items():
                times[x].append(timed(fn))
        s_old, i_old = outs["fp64_matrix_eager"]
        s_new, i_new = store.search(q, k)
        g_s, g_i = gs(q)
        r = {x: {"ms_per_call": t, "ms_per_call_median": sorted(t)[len(t) // 2]} for x, t in times.items()}
        r.update(shape=sh, same_idx=bool(torch.equal(i_old, i_new)),
                 max_abs_score_diff=float((s_old - s_new).abs().max()),
                 graph_equals_eager=bool(torch.equal(g_i, i_new) and torch.equal(g_s, s_new)))
        res[name] = r
        print(name, {x: round(r[x]["ms_per_call_median"], 4) for x in fns}, "same_idx", r["same_idx"],
              "max |ds| %.3g" % r["max_abs_score_diff"], flush=True)
        del gs, store
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except OSError:
        smi = "unavailable"
    doc = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit": smi, "steps": args.steps,
           "rounds": args.rounds, "shapes": res}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
