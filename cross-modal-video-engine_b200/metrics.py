"""Drop-in for ``LINAS-engine/util/metrics.py`` on the bit-exact rank / metric kernels (K4).

Same function names, argument meaning and return values as the reference:

* ``get_gt(video_ids, caption_ids)``            util/metrics.py:106-120  (host: it is string work)
* ``eval_q2m(scores, q2m_gts)``                 util/metrics.py:124-157
* ``t2v_map(c2i, t2v_gts)`` / ``v2t_map(...)``  util/metrics.py:61-102 + basic/metric.py:25-46
* ``t2v`` / ``v2t`` / ``*_inv_rank*``           util/metrics.py:5-57,161-218 (legacy fixed-n_caption forms)

A rank is a count (``1 + #{better}``), so the kernels stream the caller's errors matrix once instead of
sorting every row and column; R@K come from integer tallies, MedR from the rank histogram, MeanR from
the integer rank sum and AP from double-precision sums taken in rank order on the device.  The only
host arithmetic is the final ``100.0 * count / n``, ``sum / n`` and ``np.mean`` of the per-query APs,
written exactly as the reference writes them so the returned floats are identical.

Ties: the reference sorts with NumPy's default (unstable) argsort, so the order of exactly equal
scores is unspecified there; the kernels use the stable order (lower index first), i.e. the ranks are
those of ``np.argsort(line, kind="stable")``.  NaN is ordered as NumPy orders it: after every number,
NaNs by index.  A NaN ground truth (a zero embedding normalised without epsilon) is thus ranked behind
every number, not first, and a NaN element never precedes a number.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as N


def get_gt(video_ids, caption_ids):
    """Same containers, same ordering as util/metrics.py:106-120, in O(Nv + Nq) instead of O(Nv * Nq)."""
    by_video = {}
    for i, cap_id in enumerate(caption_ids):
        by_video.setdefault(cap_id.split('#', 1)[0], []).append(i)
    v2t_gt = [list(by_video.get(vid, ())) for vid in video_ids]
    t2v_gt = {}
    for i, t_gts in enumerate(v2t_gt):
        for t_gt in t_gts:
            t2v_gt.setdefault(t_gt, []).append(i)
    return v2t_gt, t2v_gt


# ---------------------------------------------------------------------------------------------------
def _csr(gts, n_query, dtype=np.int32):
    """list-of-lists / dict-by-row ground truth -> (offsets int64, ids, max per query).  C-level iteration
    (``map`` / ``chain``): 59 800 single-entry rows take ~3 ms instead of ~10 ms of Python loop."""
    from itertools import chain
    rows = [gts[i] for i in range(n_query)]          # dict: KeyError if a query has no entry, like the reference (:142)
    counts = np.fromiter(map(len, rows), dtype=np.int64, count=n_query)
    off = np.zeros(n_query + 1, dtype=np.int64)
    np.cumsum(counts, out=off[1:])
    ids = np.fromiter(chain.from_iterable(rows), dtype=dtype, count=int(off[-1]))
    return off, ids, int(counts.max()) if n_query else 0


#: lists longer than this are sorted in a global scratch buffer instead of shared memory (xmve_rank_metrics)
SORT_SMEM_ENTRIES = 16384


def rank_metrics(ranks, off, n_query, n_mem, first_only, ap_k, max_gt, best=None, ap=None, tallies=None, hist=None):
    """``xmve_rank_metrics`` with the scratch a query of more than 16384 ground-truth entries needs."""
    scratch = None
    if max_gt > SORT_SMEM_ENTRIES:
        scratch = torch.empty(ranks.numel(), dtype=torch.int32, device=ranks.device)
    N.call("xmve_rank_metrics", N.ptr(ranks), N.ptr(off), int(n_query), int(n_mem), 1 if first_only else 0, int(ap_k),
           int(max_gt), N.ptr(scratch), N.ptr(best), N.ptr(ap), N.ptr(tallies),
           N.ptr(tallies[3:]) if tallies is not None else None, N.ptr(hist), N.stream_ptr())


def _csr64(gts, n_query):
    """:func:`_csr` with int64 ids (global rows of a sharded corpus)."""
    return _csr(gts, n_query, np.int64)


def _device_matrix(scores):
    N.require_device()
    dev = torch.device("cuda", torch.cuda.current_device())
    t = scores if torch.is_tensor(scores) else torch.from_numpy(scores)
    if t.dtype not in (torch.float32, torch.float64):
        t = t.to(torch.float64)
    t = t.to(dev, non_blocking=True)
    transposed = False
    if t.dim() == 2 and t.stride(1) != 1 and t.stride(0) == 1:
        t, transposed = t.t(), True      # ``errors.T`` (validate.py:22): rank the columns of the original
    elif t.stride(1) != 1:
        t = t.contiguous()
    return t, transposed


class RankResult:
    """Device-side ranks of every ground-truth entry plus the per-query reductions."""

    def __init__(self, scores, gts, first_only=False, ap_k=0):
        x, transposed = _device_matrix(scores)
        n_row, n_col = x.shape
        axis = 1 if transposed else 0
        self.n_query = n_col if transposed else n_row
        self.n_mem = n_row if transposed else n_col
        off, ids, max_gt = _csr(gts, self.n_query)
        dev, st = x.device, N.stream_ptr()
        self.off = torch.from_numpy(off).to(dev)
        self.ids = torch.from_numpy(ids).to(dev) if ids.size else torch.zeros(1, dtype=torch.int32, device=dev)
        n_entries = int(off[-1])
        self.ranks = torch.zeros(max(n_entries, 1), dtype=torch.int32, device=dev)
        if ids.size and (ids.min() < 0 or ids.max() >= self.n_mem):
            raise IndexError("ground-truth id out of range")
        N.call("xmve_gt_ranks", N.ptr(x), N.F64 if x.dtype == torch.float64 else N.F32, n_row, n_col, x.stride(0),
               axis, N.ptr(self.off), N.ptr(self.ids), self.n_query, n_entries, max_gt, N.ptr(self.ranks), st)
        self._x = x
        self.max_gt = max_gt
        self.reduce(first_only, ap_k)

    @classmethod
    def from_store(cls, stores, queries, gts, weights=None, comm=None, n_total=None, first_only=False, ap_k=0,
                   stats=None, **kw):
        """The same ranks and reductions for a corpus whose score matrix cannot exist (SURVEY.md section 8e): the
        queries are scored against the resident (possibly sharded) ``CorpusStore`` and ``engine.rank_of_gt`` returns
        the EXACT rank of every ground-truth row -- position in the stable ascending argsort of the errors row the
        reference would form (util/metrics.py:139-145).  ``gts[i]`` lists the ground-truth GLOBAL corpus rows of
        query i (list of lists, or dict by row like ``t2v_gt``)."""
        from . import engine
        stores = list(stores) if isinstance(stores, (list, tuple)) else [stores]
        self = cls.__new__(cls)
        q = queries[0] if isinstance(queries, (list, tuple)) else queries
        self.n_query = int(q.shape[0])
        off, ids, self.max_gt = _csr64(gts, self.n_query)
        if n_total is None:
            comm_ = comm or engine.SoloComm()
            n_total = comm_.sum_int(sum(s.n for s in stores))
        self.n_mem = int(n_total)
        if ids.size and (ids.min() < 0 or ids.max() >= self.n_mem):
            raise IndexError("ground-truth id out of range")
        dev = stores[0].device
        self.off = torch.from_numpy(off).to(dev)
        self.ids = torch.from_numpy(ids).to(dev)
        ranks = engine.rank_of_gt(stores, queries, off, ids, weights=weights, comm=comm, n_total=n_total, stats=stats,
                                  **kw)
        self.ranks = ranks if ranks.numel() else torch.zeros(1, dtype=torch.int32, device=dev)
        self._x = None
        self.reduce(first_only, ap_k)
        return self

    def reduce(self, first_only=False, ap_k=0):
        dev, st = self.ranks.device, N.stream_ptr()
        self.best = torch.empty(self.n_query, dtype=torch.int32, device=dev)
        self.ap = torch.empty(self.n_query, dtype=torch.float64, device=dev)
        self.tallies = torch.zeros(4, dtype=torch.int64, device=dev)          # r<=1, r<=5, r<=10, sum of ranks
        self.hist = torch.zeros(self.n_mem + 2, dtype=torch.int32, device=dev)
        rank_metrics(self.ranks, self.off, self.n_query, self.n_mem, first_only, ap_k, self.max_gt, self.best, self.ap,
                     self.tallies, self.hist)
        return self

    def ap_vector(self, first_only=False, ap_k=0):
        """AP of every query as a device tensor, WITHOUT touching the reductions of the last :meth:`reduce` (lets
        ``cal_perf`` enqueue everything of both directions before the first device -> host read)."""
        ap = torch.empty(self.n_query, dtype=torch.float64, device=self.ranks.device)
        rank_metrics(self.ranks, self.off, self.n_query, self.n_mem, first_only, ap_k, self.max_gt, None, ap, None, None)
        return ap

    def recall_medr_meanr(self):
        n_q = self.n_query
        c1, c5, c10, rsum = (int(v) for v in self.tallies.cpu().tolist())
        r1 = 100.0 * c1 / n_q
        r5 = 100.0 * c5 / n_q
        r10 = 100.0 * c10 / n_q
        medr = _median_from_hist(self.hist.cpu().numpy(), n_q)
        meanr = np.float64(rsum) / n_q           # == int32 ranks .mean(): the fp64 sum of integers is exact
        return (r1, r5, r10, medr, meanr)

    def mean_ap(self):
        return np.mean(self.ap.cpu().numpy())


def _median_from_hist(hist, n):
    """np.median of the n integer ranks whose histogram is ``hist`` (mean of the two middle values if n is even)."""
    cum = np.cumsum(hist.astype(np.int64))
    hi = int(np.searchsorted(cum, n // 2 + 1))                  # value at sorted position n // 2
    if n % 2 == 1:
        return np.float64(hi)
    lo = int(np.searchsorted(cum, n // 2))                      # value at sorted position n // 2 - 1
    return np.float64(np.mean([lo, hi]))


def eval_q2m(scores, q2m_gts):
    """(r1, r5, r10, medr, meanr); util/metrics.py:124-157.  Pass ``errors.T`` for video->text."""
    return RankResult(scores, q2m_gts).recall_medr_meanr()


def t2v_map(c2i, t2v_gts):
    """Text->video mAP; only the FIRST ground-truth video of a caption is relevant (util/metrics.py:72-73)."""
    return RankResult(c2i, t2v_gts, first_only=True).mean_ap()


def v2t_map(c2i, v2t_gts):
    """Video->text mAP over the columns of ``c2i`` (util/metrics.py:83-102)."""
    c2i_t = c2i.T if not torch.is_tensor(c2i) else c2i.t()
    return RankResult(c2i_t, v2t_gts).mean_ap()


# ---- the same metrics, EXACT, against a resident (sharded) corpus whose score matrix cannot exist ----------------
def eval_q2m_store(stores, queries, q2m_gts, **kw):
    """``eval_q2m`` (util/metrics.py:124-157) without the matrix: exact ``(r1, r5, r10, medr, meanr)`` of the queries
    against the resident corpus.  ``**kw``: ``weights``, ``comm`` (``distributed.GroupComm``), ``n_total``."""
    return RankResult.from_store(stores, queries, q2m_gts, **kw).recall_medr_meanr()


def t2v_map_store(stores, queries, t2v_gts, **kw):
    """``t2v_map`` (util/metrics.py:61-79) without the matrix (only the FIRST ground truth counts, :72-73)."""
    return RankResult.from_store(stores, queries, t2v_gts, first_only=True, **kw).mean_ap()


def v2t_map_store(stores, queries, v2t_gts, **kw):
    """``v2t_map`` (util/metrics.py:83-102) without the matrix: the queries are the videos, the resident corpus holds
    the captions, every ground-truth caption is relevant."""
    return RankResult.from_store(stores, queries, v2t_gts, **kw).mean_ap()


# ---- the same metrics from top-k lists (approximate beyond the list: prefer the exact functions above) -----------
def eval_q2m_topk(idx, q2m_gts, n_m):
    """``eval_q2m`` (util/metrics.py:124-157) from ranked top-k lists instead of the score matrix: ``idx`` int64
    ``[n_q, k]`` from ``CorpusStore.search`` / ``sharded_search``, ``q2m_gts[i]`` the ground-truth rows of query i,
    ``n_m`` the corpus size.  A query's rank is the best position of its ground truth in the list; beyond the list it
    is only known to be ``> k``.  Returns ``(r1, r5, r10, medr, meanr, n_found)``: the recalls are exact whenever
    ``k >= 10``; ``medr`` is exact when it falls inside the lists and ``inf`` otherwise; ``meanr`` is exact only if
    every ground truth was found (``nan`` otherwise)."""
    from . import _native as N_
    from .avs import _list_ranks
    N_.require_device()
    n_q, k = idx.shape
    gts = [q2m_gts[i] for i in range(n_q)]
    off, rank, dev = _list_ranks(idx, gts, n_m)
    best = torch.empty(n_q, dtype=torch.int32, device=dev)
    tallies = torch.zeros(4, dtype=torch.int64, device=dev)
    hist = torch.zeros(n_m + 2, dtype=torch.int32, device=dev)
    rank_metrics(rank, off, n_q, n_m, False, 0, max((len(g) for g in gts), default=0), best, None, tallies, hist)
    c1, c5, c10, rsum = (int(v) for v in tallies.cpu().tolist())
    n_found = int((best <= k).sum())
    r1, r5, r10 = 100.0 * c1 / n_q, 100.0 * c5 / n_q, 100.0 * c10 / n_q
    medr = _median_from_hist(hist.cpu().numpy(), n_q)
    if medr > k:
        medr = np.float64("inf")
    meanr = np.float64(rsum) / n_q if n_found == n_q else np.float64("nan")
    return (r1, r5, r10, medr, meanr, n_found)


# ---- legacy fixed-n_caption forms (never reached from cal_perf; SURVEY.md section 8a A13) ------------
def _ranks0(c2i, gts, axis_cols):
    m = (c2i.T if not torch.is_tensor(c2i) else c2i.t()) if axis_cols else c2i
    r = RankResult(m, gts)
    return r


def _legacy_summary(ranks0):
    n = len(ranks0)
    r1 = 100.0 * len(np.where(ranks0 < 1)[0]) / n
    r5 = 100.0 * len(np.where(ranks0 < 5)[0]) / n
    r10 = 100.0 * len(np.where(ranks0 < 10)[0]) / n
    medr = np.floor(np.median(ranks0)) + 1
    meanr = ranks0.mean() + 1
    return map(float, [r1, r5, r10, medr, meanr])


def t2v(c2i, vis_details=False, n_caption=5):
    """util/metrics.py:5-29: caption i belongs to video i // n_caption; 0-based ranks."""
    assert c2i.shape[0] // c2i.shape[1] == n_caption, c2i.shape
    r = RankResult(c2i, [[i // n_caption] for i in range(c2i.shape[0])])
    return _legacy_summary(r.best.cpu().numpy().astype(np.float64) - 1)


def v2t(c2i, n_caption=5):
    """util/metrics.py:34-57: first position holding any caption of video i; 0-based ranks."""
    assert c2i.shape[0] // c2i.shape[1] == n_caption, c2i.shape
    gts = [list(range(i * n_caption, (i + 1) * n_caption)) for i in range(c2i.shape[1])]
    r = _ranks0(c2i, gts, True)
    return _legacy_summary(r.best.cpu().numpy().astype(np.float64) - 1)


def _inv_rank_mean(r):
    ranks = r.ranks.cpu().numpy()[: int(r.off[-1])].astype(np.float64)
    off = r.off.cpu().numpy()
    inv = np.zeros(r.n_query)
    for i in range(r.n_query):
        seg = np.sort(ranks[off[i]:off[i + 1]])
        inv[i] = sum(1.0 / seg)                   # the reference sums 1/(rank+1) over 0-based positions in order
    return np.mean(inv)


def t2v_inv_rank(c2i, n_caption=1):
    """util/metrics.py:161-177."""
    assert c2i.shape[0] // c2i.shape[1] == n_caption, c2i.shape
    return _inv_rank_mean(RankResult(c2i, [[i // n_caption] for i in range(c2i.shape[0])]))


def v2t_inv_rank(c2i, n_caption=1):
    """util/metrics.py:181-197."""
    assert c2i.shape[0] // c2i.shape[1] == n_caption, c2i.shape
    gts = [list(range(i * n_caption, (i + 1) * n_caption)) for i in range(c2i.shape[1])]
    return _inv_rank_mean(_ranks0(c2i, gts, True))


def v2t_inv_rank_multi(c2i, n_caption=2):
    """util/metrics.py:202-218."""
    assert c2i.shape[0] // c2i.shape[1] == n_caption, c2i.shape
    result = []
    for i in range(n_caption):
        idx = list(range(i, c2i.shape[0], n_caption))
        result.append(v2t_inv_rank(c2i[idx, :], n_caption=1))
    return result
