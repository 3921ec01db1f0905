"""Command-line front ends of the scoring path on precomputed embeddings (SURVEY.md section 8f row 3).

    python -m cross_modal_video_engine_b200.cli search --corpus DIR|video_data.pt --queries Q.npy --topK 10
        [--labels L.npy --label-mask MASK|M.npy]     (only rows whose label bit is set in the query's mask)
        [--min-score S|S.npy]                        (every row scoring at least S instead of the top K)
    python -m cross_modal_video_engine_b200.cli pairs  --corpus DIR|video_data.pt --min-score S [--out FILE]
        (every pair of corpus rows scoring at least S, each once: one line 'id_i id_j score' per pair)
    python -m cross_modal_video_engine_b200.cli eval   --corpus DIR|video_data.pt --queries Q.npy --caption-ids ids.txt
    python -m cross_modal_video_engine_b200.cli composed --index index.pt --queries queries.pt [--out results_wo_attn]

``search`` is the tail of ``LINAS-engine/inference.py:57-82`` (corpus cache -> ``cal_error`` -> ``np.argsort(...)[:topK]``
-> video ids) with the model call replaced by a file of query embeddings; with ``--run-file`` it writes a TREC run
(the AVS use of ``util/TEMPLATE_do_test_avs.sh``).  ``eval`` is the tail of ``LINAS-engine/tester.py:133-139``
(``get_gt`` -> ``cal_error`` -> ``cal_perf``, same log lines); instead of the ``pred_errors_matrix.pth.tar`` dump of
``tester.py:140`` it can save the top-k lists (``--save-topk``).  ``composed`` is the tail of
``MultiFusion/src/validate.py`` (``main`` -> ``cirr_val_retrieval`` -> ``compute_cirr_val_metrics``, :27-143) on files:
``index.pt`` = ``{"index_features": [N, 8, 640] (or pooled [N, 640]), "index_names": [N] ints}`` (what
``utils.extract_index_features`` returns) and ``queries.pt`` = ``{"predicted_features": [Nq, 640], "reference_names",
"target_names"}`` (what ``generate_cirr_val_predictions`` returns); it prints the recalls like validate.py:357-366 and
writes the top-100 names to ``<out>.npy`` like :119.  The encoders (``model.py``) are upstream of this path:
embeddings come from ``.npy`` / ``.pt`` files, a BigFile directory or the ``video_data.pt`` cache.
"""
from __future__ import annotations

import argparse
import logging
import os
import sys

import numpy as np


def _load_matrix(path):
    import torch
    if path.endswith(".npy"):
        return np.load(path)
    obj = torch.load(path, weights_only=False)
    if isinstance(obj, dict):
        obj = obj.get("embs", obj.get("video_embs", obj.get("cap_embs")))
    return obj.numpy() if hasattr(obj, "numpy") else np.asarray(obj)


def _load_corpus(path, dims):
    """-> (store, ids).  A directory is a BigFile (basic/bigfile.py), a file the video_data.pt cache."""
    from . import corpus_io
    if os.path.isdir(path):
        return corpus_io.BigFile(path).to_store(dims=dims)
    return corpus_io.load_video_data(path, dims=dims)


def _ids(path, n, prefix):
    if path is None:
        return ["%s%d" % (prefix, i) for i in range(n)]
    with open(path) as f:
        ids = f.read().split()
    if len(ids) != n:
        raise SystemExit("%s holds %d ids, expected %d" % (path, len(ids), n))
    return ids


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="cross_modal_video_engine_b200.cli", description=__doc__.split("\n\n")[0])
    sub = ap.add_subparsers(dest="cmd", required=True)
    for name in ("search", "eval"):
        p = sub.add_parser(name)
        p.add_argument("--corpus", required=True, help="BigFile directory or video_data.pt")
        p.add_argument("--queries", required=True, help=".npy / .pt matrix [Nq, D] of raw query embeddings")
        p.add_argument("--dims", default=None, help="comma-separated embedding-space dims (default: one space)")
        p.add_argument("--weights", default=None, help="comma-separated fusion weights, one per space")
        p.add_argument("--topK", type=int, default=10, help="inference.py:41")
    s = sub.choices["search"]
    s.add_argument("--query-ids", default=None)
    s.add_argument("--run-file", default=None, help="write a TREC run file instead of printing id lists")
    s.add_argument("--labels", default=None, help=".npy of one label in [0, 64) per corpus row (uint8)")
    s.add_argument("--label-mask", default=None,
                   help="search only rows whose label bit is set: one 64-bit integer, or a .npy with one per query")
    s.add_argument("--min-score", default=None,
                   help="range search: every row whose fused score is at least this (a float, or a .npy with one per "
                        "query) instead of the top K; --topK is then unused")
    pr = sub.add_parser("pairs")
    pr.add_argument("--corpus", required=True, help="BigFile directory or video_data.pt")
    pr.add_argument("--min-score", required=True, type=float, help="list every pair of rows scoring at least this")
    pr.add_argument("--dims", default=None, help="comma-separated embedding-space dims (default: one space)")
    pr.add_argument("--weights", default=None, help="comma-separated fusion weights, one per space")
    pr.add_argument("--out", default=None, help="write the pairs here instead of printing them")
    e = sub.choices["eval"]
    e.add_argument("--caption-ids", required=True, help="caption ids 'video7#enc#3' (util/metrics.py:111), one per query")
    e.add_argument("--save-topk", default=None, help="save {'scores','idx','video_ids'} of the top-K lists here")
    c = sub.add_parser("composed")
    c.add_argument("--index", required=True, help=".pt dict: index_features [N, T, D] or [N, D], index_names [N]")
    c.add_argument("--queries", required=True, help=".pt dict: predicted_features [Nq, D], reference_names, target_names")
    c.add_argument("--out", default="results_wo_attn", help="top-100 names are saved to <out>.npy (validate.py:119)")
    args = ap.parse_args(argv)
    if args.cmd == "composed":
        return args
    args.dims = tuple(int(x) for x in args.dims.split(",")) if args.dims else None
    args.weights = tuple(float(x) for x in args.weights.split(",")) if args.weights else None
    if args.dims and args.weights and len(args.dims) != len(args.weights):
        ap.error("--weights needs one value per entry of --dims")
    if args.cmd == "search" and args.label_mask is not None:
        if args.labels is None:
            ap.error("--label-mask needs --labels")
        args.label_mask = np.load(args.label_mask) if args.label_mask.endswith(".npy") else int(args.label_mask, 0)
    if args.cmd == "search" and args.min_score is not None:
        args.min_score = np.load(args.min_score) if args.min_score.endswith(".npy") else float(args.min_score)
    return args


def main(argv=None):
    args = parse_args(argv)
    if args.cmd == "composed":
        return _composed(args)
    from . import avs
    store, video_ids = _load_corpus(args.corpus, args.dims)
    if args.cmd == "pairs":
        return _pairs(args, store, video_ids)
    q = _load_matrix(args.queries)
    if args.cmd == "search":
        if args.labels is not None:
            labels = np.load(args.labels)
            store.set_labels(np.arange(store.n) + store.index_offset, labels)
        if args.min_score is not None:
            scores, idx = store.range_search(q, args.min_score, weights=args.weights,
                                             label_mask=args.label_mask).padded()
        else:
            scores, idx = store.search(q, args.topK, weights=args.weights, label_mask=args.label_mask)
        if args.run_file:
            avs.write_run_file(args.run_file, _ids(args.query_ids, len(q), "q"), idx, scores, video_ids)
        else:
            for row in idx.cpu().numpy():
                print([video_ids[i] for i in row if i >= 0])           # inference.py:80-82
        return 0
    # eval
    handler = logging.StreamHandler(sys.stdout)                         # tester.py logs its metric lines at INFO
    handler.setFormatter(logging.Formatter("%(message)s"))
    root = logging.getLogger()
    old_level = root.level
    root.addHandler(handler)
    root.setLevel(logging.INFO)
    try:
        return _eval(args, store, video_ids, q)
    finally:
        root.removeHandler(handler)
        root.setLevel(old_level)


def _eval(args, store, video_ids, q):
    import torch
    from . import evaluation, metrics, validate
    caption_ids = _ids(args.caption_ids, len(q), "cap")
    v2t_gt, t2v_gt = metrics.get_gt(video_ids, caption_ids)
    n_v = store.n
    if args.dims is None and len(q) * n_v <= (1 << 31):
        raw = store.raw[:n_v, :store.dtot].double()                     # exact fp64 path, like the reference's arrays
        errors = evaluation.cal_error(raw, torch.from_numpy(np.ascontiguousarray(q)).double())
        validate.cal_perf(errors, v2t_gt, t2v_gt)
    else:
        # the matrix cannot (or need not) exist: EXACT ranks of the ground truths against the resident corpus
        res = metrics.RankResult.from_store(store, q, t2v_gt, weights=args.weights, first_only=True)
        r1, r5, r10, medr, meanr = res.recall_medr_meanr()
        logging.info(" * Text to Video:")
        logging.info(" * r_1_5_10, medr, meanr: {}".format([round(r1, 1), round(r5, 1), round(r10, 1), round(medr, 1), round(meanr, 1)]))
        logging.info(" * recall sum: {}".format(round(r1+r5+r10, 1)))
        logging.info(" * mAP: {}".format(round(res.mean_ap(), 4)))
        logging.info(" * "+'-'*10)
    if args.save_topk:
        scores, idx = store.search(q, args.topK, weights=args.weights)
        torch.save({"scores": scores.cpu(), "idx": idx.cpu(), "video_ids": video_ids}, args.save_topk)
    return 0


def _pairs(args, store, video_ids):
    """One line ``id_i id_j score`` per pair (i < j), in the order of ``similar_pairs``: by row i, then score desc."""
    i, j, s = (t.cpu().numpy() for t in store.similar_pairs(args.min_score, weights=args.weights).pairs())
    lines = ["%s %s %r" % (video_ids[a], video_ids[b], float(c)) for a, b, c in zip(i, j, s)]
    if args.out:
        with open(args.out, "w") as f:
            f.write("".join(ln + "\n" for ln in lines))
    else:
        for ln in lines:
            print(ln)
    return 0


def _composed(args):
    import torch
    from . import multifusion
    index = torch.load(args.index, weights_only=False)
    qs = torch.load(args.queries, weights_only=False)
    feats = index["index_features"]
    feats = feats if torch.is_tensor(feats) else torch.from_numpy(np.asarray(feats))
    names = [int(x) for x in np.asarray(index["index_names"]).tolist()]
    ev = multifusion.CirrEvaluator(feats, names)
    metrics_, top = ev.metrics(qs["predicted_features"], [int(x) for x in np.asarray(qs["reference_names"]).tolist()],
                               np.asarray([int(x) for x in np.asarray(qs["target_names"]).tolist()], dtype=np.int64))
    np.save(args.out, top)
    group_recall_at1, group_recall_at2, group_recall_at3, recall_at1, recall_at5, recall_at10, recall_at50 = metrics_
    print(f"{group_recall_at1 = }")                                       # validate.py:357-363
    print(f"{group_recall_at2 = }")
    print(f"{group_recall_at3 = }")
    print(f"{recall_at1 = }")
    print(f"{recall_at5 = }")
    print(f"{recall_at10 = }")
    print(f"{recall_at50 = }")
    return 0


if __name__ == "__main__":
    sys.exit(main())
