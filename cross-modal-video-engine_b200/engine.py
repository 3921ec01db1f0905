"""Corpus-resident store and the search pipeline (host orchestration of the sm_100a kernels).

Replaces, for a corpus that is encoded once and queried many times, the per-call
``cal_error(video_embs, cap_emb)`` + ``np.argsort(errors[0])[:topK]`` of
``LINAS-engine/inference.py:78-80`` (which re-normalises the whole corpus on every call,
``evaluation.py:19-20``) and the 32-query ``1 - P @ index.T`` / ``torch.argsort`` blocks of
``MultiFusion/src/validate.py:65-113``.

The pipeline is :func:`search_shards` (its docstring lists the steps): K1 on the queries, a sampled per-query
threshold, the fused tcgen05 score + threshold filter over the resident operand (the score matrix never reaches
HBM), an exact fp64 rescore of the survivors in two rounds, a bitonic top-k with a certificate that nothing
outside the candidate set can belong to the top-k, and a re-run of the rare rows that miss the certificate.
The first pass never waits for the host: the error bound is a device scalar, the number of uncertified rows comes
back through one asynchronous copy (``defer=True`` hands the caller a :class:`PendingSearch` to resolve later).
:meth:`CorpusStore.search` is the one-shard case; ``distributed.sharded_search`` joins the shards of several GPUs.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import struct

import torch

from . import _native as N

#: former fallback bound per unit of fusion weight (2 * 2^-8 plus accumulation slack for rows up to K ~ 2800); it stays
#: the floor of :func:`eps_fallback`, which raises it to the a-priori bound where the accumulation term needs more
EPS_X1 = 8.5e-3
SMALL_NV = 16384
#: multiples of eps subtracted from the sampled threshold kth(sample, j) -- see :func:`thr_margin`.  Round 1 always
#: used 2: "the k-th best exact score is at least kth_approx - eps, a row's approximate score at most eps above its
#: exact one".  But j already carries a 5.5-sigma sampling slack (plan()): the j-th largest of the sample sits near
#: corpus rank j * step (1 500 at C5), an order of magnitude below the k-th best, so the certificate
#: kth_exact - eps >= thr holds without the extra margin (P(miss) ~ 1e-7 per row; a miss only costs a re-run of that
#: row).  Dropping it cuts the candidate lists from 5 800 to 1 500 per query at C5 and from 2 350 to 1 200 at C4.
THR_EPS_MARGIN = 0.0


def thr_margin(lam):
    """Multiples of eps to subtract from ``kth(sample, j)`` for ``lam = k / step`` expected top-k rows in the sample.

    The margin-free threshold lives on the score gap between corpus rank ``k`` and rank ``j * step``.  The rank ratio
    ``j / lam = 1 + 5.5 / sqrt(lam) + 4 / lam`` is >= 3.3 for ``lam <= 8.5`` (a gap of ~0.4 sigma of the score
    distribution against eps ~ 0.2 sigma) but tends to 1 for deep lists over small corpora (k = 1000 of 200 k rows:
    1.9), where the missing margin showed up as re-runs -- a whole extra FILTER pass for the rows concerned
    (profiles/r2_summary.md section 6).  So: none up to lam = 8.5, one eps up to 64, the rigorous two beyond.  A wrong
    guess costs time, never correctness (the certificate decides)."""
    if lam <= 8.5:
        return THR_EPS_MARGIN
    return max(THR_EPS_MARGIN, 1.0 if lam <= 64.0 else 2.0)
ROW_TOPJ_MAX = 4096
#: size of the strided corpus sample that sets the per-query threshold: n / SAMPLE_DIV rows, clamped to
#: [SAMPLE_MIN, SAMPLE_MAX] (plan()).  A larger sample costs a longer sampling pass and buys a tighter threshold,
#: i.e. fewer candidates for the FILTER epilogue, the order statistics and the rescore.
SAMPLE_DIV = int(os.environ.get("XMVE_SAMPLE_DIV", 128))
SAMPLE_MIN = int(os.environ.get("XMVE_SAMPLE_MIN", 8192))
SAMPLE_MAX = int(os.environ.get("XMVE_SAMPLE_MAX", 65536))
_BM, _BN = 128, 256
#: corpus row labels are 0 .. N_LABELS - 1: one byte per row, one 64-bit mask per query (filtered search)
N_LABELS = 64


def _round_up(x, m):
    return (x + m - 1) // m * m


def _as_spaces(x, dims):
    """Split ``x`` (tensor ``[n, sum(dims)]`` / ``[n, T, sum(dims)]`` or a per-space list) into per-space views."""
    if isinstance(x, (list, tuple)):
        assert len(x) == len(dims), "expected one array per embedding space"
        return list(x)
    if len(dims) == 1:
        return [x]
    out, o = [], 0
    for d in dims:
        out.append(x[..., o:o + d])
        o += d
    return out


def _to_device(x, device):
    """numpy / torch, host / device -> CUDA tensor (fp32 or fp64), last dim contiguous."""
    if not torch.is_tensor(x):
        import numpy as np
        x = torch.from_numpy(np.ascontiguousarray(x))
    if x.dtype not in (torch.float32, torch.float64):
        x = x.float()
    x = x.to(device, non_blocking=True)
    return x


def _host_ints(x):
    """ids / labels from a tensor, ndarray, sequence or scalar -> int64 CPU tensor."""
    if torch.is_tensor(x):
        return x.detach().to("cpu", torch.int64)
    import numpy as np
    return torch.from_numpy(np.asarray(x).astype(np.int64))


def _check_labels(labels, n, device):
    """``n`` row labels in [0, N_LABELS) -> int64 tensor on ``device``; ValueError otherwise."""
    lab = _host_ints(labels).flatten()
    if lab.numel() != n:
        raise ValueError("expected %d labels, got %d" % (n, lab.numel()))
    if lab.numel() and (int(lab.min()) < 0 or int(lab.max()) >= N_LABELS):
        raise ValueError("labels must lie in [0, %d)" % N_LABELS)
    return lab.to(device)


def _label_masks(label_mask, nq, device):
    """``search(label_mask=...)`` -> int64 device tensor ``[nq]`` holding the 64-bit masks (uint64 bit patterns)."""
    if torch.is_tensor(label_mask):
        m = label_mask
        if m.dtype not in (torch.int64, torch.uint64):
            raise ValueError("label_mask: expected an int64 or uint64 tensor, got %s" % m.dtype)
        m = m.view(torch.int64) if m.dtype == torch.uint64 else m
    else:
        import numpy as np
        a = np.asarray(label_mask)                     # a Python int of 2^63 or more comes out as uint64
        if a.dtype == np.uint64:
            a = a.view(np.int64)
        elif a.dtype.kind == "i":
            a = a.astype(np.int64)
        else:
            raise ValueError("label_mask: expected 64-bit integer masks, got %s" % a.dtype)
        m = torch.from_numpy(np.ascontiguousarray(a))
    if m.dim() == 0 or m.numel() == 1:
        m = m.reshape(1).expand(nq)
    if tuple(m.shape) != (nq,):
        raise ValueError("label_mask: expected one mask per query (%d) or one for all, got shape %s"
                         % (nq, tuple(m.shape)))
    return m.to(device, non_blocking=True).contiguous()


def _eligible_counts(masks, hist):
    """``n_elig[q] = sum over the set bits l of masks[q] of hist[l]`` on the device (no host round trip)."""
    bits = torch.bitwise_and(torch.bitwise_right_shift(masks.unsqueeze(1),
                                                       torch.arange(N_LABELS, device=masks.device)), 1)
    return (bits * hist.unsqueeze(0)).sum(1)


def _prepare(src, d, raw, raw_off, norm, resid, op, op_off, layout, weight, norm_mode):
    """One K1 launch for one embedding space of one batch of rows."""
    frames = 1
    if src.dim() == 3:
        frames = src.shape[1]
    n = src.shape[0]
    if n == 0:
        return
    if src.stride(-1) != 1 or (frames > 1 and src.stride(1) != d):
        src = src.contiguous()
    if frames > 1 and not src.is_contiguous():
        src = src.contiguous()
    N.call("xmve_prepare_rows", N.ptr(src), N.F64 if src.dtype == torch.float64 else N.F32, n, d, frames,
           src.stride(0),
           N.ptr(raw), raw.stride(0) if raw is not None else 0, raw_off,
           N.ptr(norm), N.ptr(resid),
           N.ptr(op), op.stride(0) if op is not None else 0, op_off, layout,
           float(weight), norm_mode, N.stream_ptr())


class CorpusStore:
    """Video-embedding corpus resident in HBM: bf16 operand rows + raw fp32 rows + fp64 norms.

    ``dims`` lists the embedding spaces (e.g. ``(1536, 512)`` for latent + concept); rows are appended
    with :meth:`add` (the analogue of ``encode_vid``'s batch loop, evaluation.py:98-105) and
    normalised once, on the device, as they arrive.  ``index_offset`` is this shard's first global
    row (multi-GPU sharding).

    Memory: ``capacity * (2 * sum(dpad) + 4 * sum(dims) + 12 * S)`` bytes -- 12.3 KB per row at 1536 + 512 dims, i.e.
    123 GB for the 10 M-row C5 corpus (41 GB bf16 operand + 82 GB fp32 raw rows kept for the exact rescore) and a
    ceiling of about 14 M such rows per 180 GB B200; larger corpora are sharded (``distributed.shard_range``).  The
    constructor checks the free device memory first and raises a sized ``MemoryError`` instead of a CUDA OOM.

    Inputs are taken as the reference keeps them: fp32 model outputs, possibly stored in float64 arrays
    (evaluation.py:102-105).  float64 inputs are therefore narrowed to fp32 by K1 (exact for such arrays); the
    fp64 arithmetic of the rescore then equals ``cal_error`` on the float64 copies.  Genuinely double-precision
    embeddings would be ranked after rounding to fp32 -- use ``evaluation.cal_error`` for those.
    """

    def __init__(self, capacity, dims, device="cuda", norm_mode="plain", index_offset=0):
        N.require_device()
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.dims = tuple(int(d) for d in (dims if isinstance(dims, (list, tuple)) else (dims,)))
        self.dpads = tuple(_round_up(d, 64) for d in self.dims)
        self.k = sum(self.dpads)
        self.dtot = sum(self.dims)
        self.raw_ld = _round_up(self.dtot, 4)
        self.capacity = int(capacity)
        self.norm_mode = {"plain": N.NORM_PLAIN, "eps": N.NORM_EPS}[norm_mode]
        self.index_offset = int(index_offset)
        self.n = 0
        rows = _round_up(max(self.capacity, 1), _BN)
        need = rows * self.k * 2 + max(self.capacity, 1) * (self.raw_ld * 4 + len(self.dims) * 12)
        free = torch.cuda.mem_get_info(self.device)[0] + torch.cuda.memory_reserved(self.device) \
            - torch.cuda.memory_allocated(self.device)
        if need > free:
            raise MemoryError(
                "CorpusStore: %d rows x %s dims need %.1f GB of HBM (bf16 operand + fp32 raw rows + norms) but only "
                "%.1f GB are free on %s; shard the corpus over more GPUs (distributed.shard_range) or lower the "
                "capacity" % (self.capacity, list(self.dims), need / 1e9, free / 1e9, self.device))
        self.op = torch.zeros((rows, self.k), dtype=torch.bfloat16, device=self.device)
        self.raw = torch.empty((max(self.capacity, 1), self.raw_ld), dtype=torch.float32, device=self.device)
        self.norm = torch.empty((len(self.dims), max(self.capacity, 1)), dtype=torch.float64, device=self.device)
        self.resid = torch.zeros((len(self.dims), max(self.capacity, 1)), dtype=torch.float32, device=self.device)
        self._resid_max2 = None
        self.added = None                                     # CUDA event after the last add's kernels
        # label plane (uint8 per row, 0 <= label < N_LABELS) and the device histogram of the filled rows' labels;
        # allocated on first use (add(..., labels) / set_labels / a filtered search)
        self.labels = None
        self.label_hist = None
        self.label_version = 0                                # bumped by set_labels (GraphSearch checks it)
        self.space_off = (C.c_int32 * (len(self.dims) + 1))(*([0] + list(_cumsum(self.dims))))

    # -- ingest ----------------------------------------------------------------------------------
    def add(self, rows, labels=None):
        """Append rows: tensor / ndarray ``[n, sum(dims)]`` (or ``[n, T, D]``: mean over T first), or a per-space list.
        ``labels`` (``n`` integers in ``[0, 64)``, see ``search(label_mask=...)``) label the new rows; rows added
        without labels have label 0."""
        spaces = [_to_device(s, self.device) for s in _as_spaces(rows, self.dims)]
        n = spaces[0].shape[0]
        if self.n + n > self.capacity:
            raise ValueError("CorpusStore capacity %d exceeded" % self.capacity)
        if labels is not None:
            labels = _check_labels(labels, n, self.device)
        op_off = raw_off = 0
        with torch.cuda.device(self.device):                  # launch on the store's device, whatever is current
            for s, (src, d, dp) in enumerate(zip(spaces, self.dims, self.dpads)):
                assert src.shape[-1] == d, "space %d: expected dim %d, got %d" % (s, d, src.shape[-1])
                _prepare(src, d, self.raw[self.n:], raw_off, self.norm[s, self.n:], self.resid[s, self.n:],
                         self.op[self.n:], op_off, N.OP_X1, 1.0, self.norm_mode)
                op_off += dp
                raw_off += d
            if labels is not None or self.labels is not None:
                self._ensure_labels()
                if labels is not None:
                    self.labels[self.n:self.n + n] = labels.to(torch.uint8)
                    self.label_hist += torch.bincount(labels, minlength=N_LABELS)
                else:
                    self.labels[self.n:self.n + n] = 0
                    self.label_hist[0] += n
            # a search's head stream (search_shards(head_stream=...)) reads the new rows: it waits for this event
            self.added = torch.cuda.Event()
            self.added.record()
        self.n += n
        return self

    def set_labels(self, ids, labels):
        """Relabel rows: ``ids`` are global row numbers (as :meth:`search` returns them), ``labels`` one integer in
        ``[0, 64)`` per id.  The store applies the ids that fall in its rows ``[index_offset, index_offset + n)`` and
        skips the others, which belong to other shards.  A search issued afterwards, on any stream, sees the new
        labels.

        For a corpus sharded over several stores or ranks this is a collective call: every shard is given the same
        ``ids`` and ``labels``, even when none of them is its own.  The searches of all ranks then agree on the label
        state, whose global histogram they all-reduce once per change."""
        ids = torch.as_tensor(_host_ints(ids), dtype=torch.int64).flatten()
        if ids.numel() and int(ids.min()) < 0:
            raise IndexError("set_labels: negative row id")
        if torch.unique(ids).numel() != ids.numel():
            raise ValueError("set_labels: duplicate ids")
        labels = _check_labels(labels, ids.numel(), self.device)
        loc = ids - self.index_offset
        mine = (loc >= 0) & (loc < self.n)
        loc, labels = loc[mine], labels[mine.to(labels.device)]
        with torch.cuda.device(self.device):
            self._ensure_labels()
            loc = loc.to(self.device)
            self.label_hist -= torch.bincount(self.labels[loc].long(), minlength=N_LABELS)
            self.labels[loc] = labels.to(torch.uint8)
            self.label_hist += torch.bincount(labels, minlength=N_LABELS)
            self.added = torch.cuda.Event()                   # head-stream searches wait for the new labels
            self.added.record()
        self.label_version += 1
        return self

    def _ensure_labels(self):
        """Allocate the label plane (every row label 0) and its histogram on first use."""
        if self.labels is None:
            self.labels = torch.zeros((max(self.capacity, 1),), dtype=torch.uint8, device=self.device)
            self.label_hist = torch.zeros((N_LABELS,), dtype=torch.int64, device=self.device)
            self.label_hist[0] = self.n
        return self.labels

    def _label_counts(self):
        """int64 [64]: how many filled rows carry each label (device)."""
        self._ensure_labels()
        return self.label_hist

    # -- query side ------------------------------------------------------------------------------
    def prepare_queries(self, queries, weights=None):
        """K1 on the query batch: returns (a_op bf16 [nq_pad, K], q_raw fp32 [nq, raw_ld], q_norm fp64 [S, nq],
        q_resid fp32 [S, nq] squared bf16 residuals, nq)."""
        weights = _weights(weights, len(self.dims))
        spaces = [_to_device(s, self.device) for s in _as_spaces(queries, self.dims)]
        nq = spaces[0].shape[0]
        a_op = torch.zeros((_round_up(max(nq, 1), _BM), self.k), dtype=torch.bfloat16, device=self.device)
        q_raw = torch.empty((max(nq, 1), self.raw_ld), dtype=torch.float32, device=self.device)
        q_norm = torch.empty((len(self.dims), max(nq, 1)), dtype=torch.float64, device=self.device)
        q_res = torch.zeros((len(self.dims), max(nq, 1)), dtype=torch.float32, device=self.device)
        op_off = raw_off = 0
        for s, (src, d, dp) in enumerate(zip(spaces, self.dims, self.dpads)):
            _prepare(src, d, q_raw, raw_off, q_norm[s], q_res[s], a_op, op_off, N.OP_X1, weights[s], self.norm_mode)
            op_off += dp
            raw_off += d
        return a_op, q_raw, q_norm, q_res, nq

    # -- search ----------------------------------------------------------------------------------
    def search(self, queries, k, weights=None, exclude=None, eps=None, small_nv=SMALL_NV, stats=None, defer=False,
               label_mask=None):
        """Top-``k`` corpus rows per query by fused cosine score, exact (fp64) scores, descending.

        Returns ``(scores float64 [nq, k], idx int64 [nq, k])`` on the device; ``idx`` are global row
        numbers (``index_offset`` + local), ``-1`` / ``-inf`` padded if the corpus has fewer than ``k``
        rows.  ``exclude[q]`` (global row or -1) is dropped from row q's list -- MultiFusion's removal
        of the query's own reference item (validate.py:76-83).  ``eps`` overrides the measured bound on
        |tensor-core score - exact score| (see :func:`measured_eps`).  ``defer=True`` returns a
        :class:`PendingSearch` as soon as the work is enqueued (``.result()`` gives the tuple).

        ``label_mask`` (filtered search): one 64-bit mask per query (int64 / uint64 tensor or array ``[nq]``) or one
        for the whole batch.  Row ``v`` is eligible for query ``q`` iff bit ``label[v]`` of ``mask[q]`` is set
        (labels: :meth:`add`, :meth:`set_labels`); the result is the exact top-``min(k, #eligible)`` of the eligible
        rows, padded as above.  ``None`` searches every row.
        """
        return search_shards([self], queries, k, weights=weights, exclude=exclude, eps=eps, small_nv=small_nv,
                             stats=stats, defer=defer, label_mask=label_mask)

    def range_search(self, queries, min_score, weights=None, exclude=None, label_mask=None, eps=None, stats=None):
        """Every corpus row whose exact fused score reaches ``min_score`` (a float, or one per query), per query,
        sorted by (score desc, global row asc) -> :class:`RangeResult`.  Scores are the fp64 scores :meth:`search`
        returns; the lists are complete.  ``+inf`` gives an empty list, ``-inf`` every eligible row.  ``exclude`` and
        ``label_mask`` as in :meth:`search`.  A result too large for the free device memory raises a sized
        ``MemoryError`` before it is allocated (:meth:`range_count` counts without listing)."""
        return range_search_shards([self], queries, min_score, weights=weights, exclude=exclude,
                                   label_mask=label_mask, eps=eps, stats=stats)

    def range_count(self, queries, min_score, weights=None, exclude=None, label_mask=None, eps=None):
        """int64 ``[nq]`` on the device: the length of each :meth:`range_search` list for the same arguments, without
        listing the rows -- only the rows within the error bound of ``min_score`` are listed and rescored."""
        return range_count_shards([self], queries, min_score, weights=weights, exclude=exclude,
                                  label_mask=label_mask, eps=eps)

    def similar_pairs(self, min_score, weights=None, eps=None, stats=None):
        """Every pair of stored rows ``i < j`` whose exact fused score reaches ``min_score`` (one float), each pair once
        -> :class:`RangeResult` with one list per row ``i``: the rows ``j > i`` with ``s(i, j) >= min_score``, sorted
        by (score desc, j asc).  ``s(i, j)`` is the fp64 score :meth:`range_search` gives row ``j`` for the stored
        row ``i`` as the query.  ``+inf`` gives no pairs, ``-inf`` every pair; NaN raises ``ValueError``.
        :meth:`RangeResult.pairs` gives the COO form.  See :func:`similar_pairs_shards`."""
        return similar_pairs_shards([self], min_score, weights=weights, eps=eps, stats=stats)

    def _suffix(self, start):
        """This store's rows ``[start, n)`` as a store of their own, without copies (global rows keep their numbers):
        operand, raw rows, norm and residual planes and labels offset by ``start``.  The norm planes keep their
        ``[S, capacity]`` row stride, which is what the rescore reads; the operand's row stride is a multiple of 128 B,
        so its tensor map may start at any row.  The error bound reads this store's residuals over EVERY row."""
        start = min(int(start), self.n)
        v = object.__new__(type(self))
        v.__dict__.update(self.__dict__)
        v.op, v.raw = self.op[start:], self.raw[start:]
        v.norm, v.resid = self.norm[:, start:], self.resid[:, start:]
        v.labels = None if self.labels is None else self.labels[start:]
        v.n, v.capacity, v.index_offset = self.n - start, self.capacity - start, self.index_offset + start
        v.resid_max2 = self.resid_max2
        v._dv2_cache = None                                   # (keyed by row counts: a view's must not hit it)
        return v

    def plan(self, k, n=None):
        return plan(k, self.n if n is None else n)

    def resid_max2(self):
        """max over rows of the squared bf16 quantisation residual of the operand (device scalar, cached)."""
        if self._resid_max2 is None or self._resid_max2[0] != self.n:
            r = self.resid[:, :self.n].sum(0).max() if self.n else torch.zeros((), device=self.device)
            self._resid_max2 = (self.n, r)
        return self._resid_max2[1]

    def _weights_arr(self, wts):
        return (C.c_double * len(wts))(*[float(w) for w in wts])

    def _exact_small(self, q_raw, q_norm, nq, k, wts, excl, label_mask=None):
        """fp64 score matrix + bitonic top-k (corpora up to ``small_nv`` rows); ``label_mask``: ineligible rows are
        set to -inf first, and the selection skips them."""
        dev, st = self.device, N.stream_ptr()
        acc = None
        o = 0
        for s, d in enumerate(self.dims):
            qn = torch.empty((nq, d), dtype=torch.float64, device=dev)
            vn = torch.empty((self.n, d), dtype=torch.float64, device=dev)
            qs, vs = q_raw[:nq, o:o + d], self.raw[:self.n, o:o + d]
            N.call("xmve_normalize_f64", N.ptr(qs), N.F32, nq, d, q_raw.stride(0), N.ptr(qn), d, self.norm_mode, st)
            N.call("xmve_normalize_f64", N.ptr(vs), N.F32, self.n, d, self.raw.stride(0), N.ptr(vn), d,
                   self.norm_mode, st)
            sc = torch.empty((nq, self.n), dtype=torch.float64, device=dev)
            for q0 in range(0, nq, 1 << 21):
                q1 = min(nq, q0 + (1 << 21))
                N.call("xmve_score_f64", N.ptr(qn[q0:]), q1 - q0, d, N.ptr(vn), self.n, d, d, float(wts[s]),
                       N.ptr(sc[q0:]), self.n, st)
            acc = sc if acc is None else acc.add_(sc)
            o += d
        if label_mask is not None:
            N.call("xmve_mask_scores", N.ptr(acc), N.F64, nq, self.n, acc.stride(0), N.ptr(self._ensure_labels()), 1,
                   N.ptr(label_mask), st)
        kk = min(k, self.n)
        out_s = torch.full((nq, k), float("-inf"), dtype=torch.float64, device=dev)
        out_i = torch.full((nq, k), -1, dtype=torch.int64, device=dev)
        s_ = torch.empty((nq, kk), dtype=torch.float64, device=dev)
        i_ = torch.empty((nq, kk), dtype=torch.int64, device=dev)
        N.call("xmve_select_topk_i32", N.ptr(acc), None, nq, self.n, None, self.index_offset, N.ptr(excl), kk,
               None, 0.0, None, None, N.ptr(s_), N.ptr(i_), None, None, None, None, st)
        out_s[:, :kk] = s_
        out_i[:, :kk] = i_
        return out_s, out_i

    # one shard's share of a filtered pass ----------------------------------------------------------
    def _sample(self, a_op, nq, step, label_mask=None):
        """K2 STORE over every ``step``-th row of this shard -> fp32 ``[nq, ceil(n / step)]`` (``label_mask``: -inf
        where the sampled row is not eligible)."""
        n_s = (self.n + step - 1) // step
        sample = torch.empty((nq, n_s), dtype=torch.float32, device=self.device)
        N.call("xmve_score_store", N.ptr(a_op), nq, a_op.stride(0), N.ptr(self.op), n_s, self.op.stride(0), step,
               self.k, 1.0, N.ptr(sample), sample.stride(0), N.stream_ptr())
        if label_mask is not None:
            N.call("xmve_mask_scores", N.ptr(sample), N.F32, nq, n_s, sample.stride(0), N.ptr(self._ensure_labels()),
                   step, N.ptr(label_mask), N.stream_ptr())
        return sample

    def _filter(self, a_op, nq, thr, cap, step=1, label_mask=None):
        """K2 FILTER over the shard (or over every ``step``-th row): candidates (approximate score, local row --
        sampled-row number when ``step > 1``) above ``thr`` per query; ``label_mask``: eligible rows only."""
        dev = self.device
        rows = (self.n + step - 1) // step
        cand_count = torch.zeros((nq,), dtype=torch.int32, device=dev)
        cand_score = torch.empty((nq, cap), dtype=torch.float32, device=dev)
        cand_idx = torch.empty((nq, cap), dtype=torch.int32, device=dev)
        if label_mask is not None:
            N.call("xmve_score_filter_labeled", N.ptr(a_op), nq, a_op.stride(0), N.ptr(self.op), rows,
                   self.op.stride(0), step, self.k, N.ptr(thr), None, None, N.ptr(cand_count), N.ptr(cand_score),
                   N.ptr(cand_idx), cap, N.ptr(self._ensure_labels()), N.ptr(label_mask), N.stream_ptr())
            return cand_count, cand_score, cand_idx
        N.call("xmve_score_filter", N.ptr(a_op), nq, a_op.stride(0), N.ptr(self.op), rows, self.op.stride(0), step,
               self.k, N.ptr(thr), None, None, N.ptr(cand_count), N.ptr(cand_score), N.ptr(cand_idx), cap,
               N.stream_ptr())
        return cand_count, cand_score, cand_idx

    def _filter_band(self, a_op, nq, lo, hi, cap, label_mask=None):
        """K2 FILTER with a two-sided window per row: rows scoring above ``hi`` are counted, rows in ``(lo, hi]``
        are listed -> (above int32 [nq], count int32 [nq], scores fp32 [nq, cap], local rows int32 [nq, cap]).
        ``label_mask``: eligible rows only, counted and listed."""
        dev = self.device
        above = torch.zeros((nq,), dtype=torch.int32, device=dev)
        count = torch.zeros((nq,), dtype=torch.int32, device=dev)
        c_s = torch.empty((nq, cap), dtype=torch.float32, device=dev)
        c_i = torch.empty((nq, cap), dtype=torch.int32, device=dev)
        if label_mask is not None:
            N.call("xmve_score_filter_labeled", N.ptr(a_op), nq, a_op.stride(0), N.ptr(self.op), self.n,
                   self.op.stride(0), 1, self.k, N.ptr(lo), N.ptr(hi), N.ptr(above), N.ptr(count), N.ptr(c_s),
                   N.ptr(c_i), cap, N.ptr(self._ensure_labels()), N.ptr(label_mask), N.stream_ptr())
            return above, count, c_s, c_i
        N.call("xmve_score_filter", N.ptr(a_op), nq, a_op.stride(0), N.ptr(self.op), self.n, self.op.stride(0), 1,
               self.k, N.ptr(lo), N.ptr(hi), N.ptr(above), N.ptr(count), N.ptr(c_s), N.ptr(c_i), cap, N.stream_ptr())
        return above, count, c_s, c_i

    def _sample_top(self, a_op, nq, step, big_j, label_mask=None):
        """The largest scores of the ``step``-strided sample of this shard WITHOUT writing the sample matrix:
        a coarse STORE pass (every ``r * step``-th row, a few thousand columns) gives a per-query floor ``thr0``
        that about ``4 * big_j`` of the fine sample's scores exceed; a FILTER pass over the fine sample keeps those.
        Returns ``(scores fp32 [nq, cap_s], counts int32 [nq], thr0 fp32 [nq])``; rows whose count is below
        ``big_j`` (the floor came out too high -- vanishingly rare) are handled by the caller through ``thr0``.
        ``label_mask``: both passes see the eligible rows only."""
        n_s = (self.n + step - 1) // step
        r = max(2, min(16, n_s // 2048))
        kw = {} if label_mask is None else {"label_mask": label_mask}
        coarse = self._sample(a_op, nq, step * r, **kw)
        j0 = min(coarse.shape[1], int(math.ceil(4.0 * big_j / r)))
        thr0 = _row_kth(coarse, None, j0, 0.0, 0)
        cap_s = 1 << max(10, int(math.ceil(math.log2(16 * big_j))))
        count, score, _ = self._filter(a_op, nq, thr0, cap_s, step=step, **kw)
        return score, count, thr0

    def _rescore(self, q_raw, q_norm, nq, wts, cand, bound, bound_hi=None, exact=None):
        """Exact fp64 scores of the candidates whose approximate score reaches ``bound`` (second round: of those in
        ``[bound, bound_hi)``, the entries at or above ``bound_hi`` keep their first-round values) -> fp64 [nq, cap]."""
        cand_count, cand_score, cand_idx = cand
        cap = cand_score.shape[1]
        if exact is None:
            exact = torch.empty((nq, cap), dtype=torch.float64, device=self.device)
        # the norm planes are [S, capacity]: their row stride, not the number of rows filled, locates space s
        N.call("xmve_rescore", N.ptr(q_raw), nq, q_raw.stride(0), N.ptr(q_norm), N.ptr(self.raw), self.norm.stride(0),
               self.raw.stride(0), N.ptr(self.norm), len(self.dims), self.space_off, self._weights_arr(wts),
               self.norm_mode, N.ptr(cand_score), N.ptr(cand_idx), N.ptr(cand_count), cap, N.ptr(bound),
               N.ptr(bound_hi), N.ptr(exact), N.stream_ptr())
        return exact

    def _pilot_top(self, exact, cand, nq, excl, m):
        """The ``m`` largest first-round exact scores per query, descending, -inf padded -> fp64 [nq, m]."""
        cand_count, cand_score, cand_idx = cand
        out = torch.empty((nq, m), dtype=torch.float64, device=self.device)
        N.call("xmve_pilot_top", N.ptr(exact), N.ptr(cand_idx), N.ptr(cand_count), nq, cand_score.shape[1],
               self.index_offset, N.ptr(excl), m, N.ptr(out), N.stream_ptr())
        return out

    def _select(self, exact, cand, nq, k, excl, thr, eps_t, bound, out_s, out_i, certify, n_bad=None):
        """Local top-k (global row ids) of the rescored candidates into ``out_s`` / ``out_i`` -> ``(cert, thr_next)``.
        ``certify=False`` (a shard's list for the merge): ``cert`` says whether the list is exact -- 0 after a
        candidate-list overflow or when more float-tied scores than the sort holds had to be cut -- and ``thr_next``
        is None."""
        cand_count, cand_score, cand_idx = cand
        cap = cand_score.shape[1]
        thr_next = None
        cert = torch.empty((nq,), dtype=torch.int32, device=self.device)
        if certify:
            thr_next = torch.empty((nq,), dtype=torch.float32, device=self.device)
        N.call("xmve_select_topk_i32", N.ptr(exact), N.ptr(cand_idx), nq, cap, N.ptr(cand_count),
               self.index_offset, N.ptr(excl), k, N.ptr(thr) if certify else None, 1.0, N.ptr(eps_t),
               N.ptr(bound) if certify else None, N.ptr(out_s), N.ptr(out_i), None, N.ptr(cert), N.ptr(thr_next),
               N.ptr(n_bad) if certify else None, N.stream_ptr())
        return cert, thr_next


def plan(k, n):
    """Sampling step, order statistics and candidate capacity for a top-``k`` search of ``n`` corpus rows."""
    n = int(n)
    n_s = min(n, max(SAMPLE_MIN, min(SAMPLE_MAX, n // SAMPLE_DIV)))
    step = max(1, n // max(n_s, 1))
    n_s = (n + step - 1) // step
    lam = k / step
    j = int(math.ceil(lam + 5.5 * math.sqrt(lam) + 4))
    cap = 1 << max(11, int(math.ceil(math.log2(8 * step * j))))
    cap = min(cap, 32768)
    j_cap = max(j, int(0.5 * cap / step))
    return {"step": step, "n_sample": n_s, "j": min(j, n_s), "j_cap": min(j_cap, n_s), "cap": cap,
            "margin": thr_margin(lam)}


def measured_eps(dq, dv, wts, n_space, k_len):
    """Rigorous bound on |tensor-core score - exact score| from the MEASURED bf16 residuals.

    With Q = concat_s(w_s q_hat_s), V = concat_s(v_hat_s) and Qb, Vb their bf16 roundings,
    ``<Q,V> - <Qb,Vb> = <Q-Qb, V> + <Qb, V-Vb>``, so by Cauchy-Schwarz the operand rounding costs at most
    ``dq * |V| + |Qb| * dv`` with ``dq = max_q |Q-Qb|``, ``dv = max_v |V-Vb|`` (K1 measures both), ``|V| = sqrt(S)``
    and ``|Qb| <= sqrt(sum w^2) + dq``.  The bf16 x bf16 products are exact in fp32; accumulating ``k_len`` of them
    in fp32 (with truncation at worst) costs at most ``k_len * 2^-22 * |Qb| * |Vb|``.  Without measurements the bound
    is :func:`eps_fallback`; Gaussian-like rows measure ``dq, dv ~ 1.7e-3`` of the norm, about half the worst case.
    """
    qn = math.sqrt(sum(w * w for w in wts)) + dq
    vn = math.sqrt(n_space) * (1.0 + 2.0 ** -8)
    e = dq * vn + qn * dv + k_len * 2.0 ** -22 * qn * vn + 1e-6
    if not math.isfinite(e) or e <= 0.0:                   # NaN rows (zero vectors under 'plain' normalisation)
        return eps_fallback(wts, n_space, k_len)
    return e


def eps_fallback(wts, n_space, k_len):
    """Bound on |tensor-core score - exact score| that needs no measured residual; used when a residual is NaN.

    bf16 keeps 8 significant bits, so rounding moves each space's operand by at most ``u = 2^-8`` of its norm: the
    product of space ``s`` moves by at most ``|w_s| * (2u + u^2)`` (Cauchy-Schwarz, both sides).  Accumulating
    ``k_len`` products in fp32 adds ``k_len * 2^-22 * |Qb| * |Vb|`` with ``|Qb| <= |w| (1 + u)`` and
    ``|Vb| <= sqrt(S) (1 + u)``; ``1e-6`` covers the fp32 rounding of the operand before its bf16 rounding.  The
    accumulation term grows with ``k_len``, so no constant per unit weight bounds every layout: ``EPS_X1`` alone fell
    below it from K = 2816 on.  Returns the larger of ``EPS_X1 * max(1, sum |w|)`` (unchanged where it was sound) and
    that bound, as the smallest fp32 value at or above it, since the device takes it as a float."""
    u = 2.0 ** -8
    e = (sum(abs(w) for w in wts) * (2 * u + u * u)
         + k_len * 2.0 ** -22 * math.sqrt(sum(w * w for w in wts)) * (1 + u) * math.sqrt(n_space) * (1 + u) + 1e-6)
    e = max(e, EPS_X1 * max(1.0, sum(abs(w) for w in wts)))
    e *= 1 + 1e-12                                          # the float64 evaluation above rounds either way
    f = struct.unpack("<f", struct.pack("<f", e))[0]         # nearest fp32
    if f < e:
        f = struct.unpack("<f", struct.pack("<I", struct.unpack("<I", struct.pack("<f", f))[0] + 1))[0]
    return f


class _Phases:
    """CUDA-event marks at the phase boundaries of a search (only when the caller passes ``stats``)."""

    def __init__(self, on):
        self.on, self.marks = on, []

    def mark(self, name):
        if self.on:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.marks.append((name, e))

    def result(self):
        if len(self.marks) < 2:
            return {}
        self.marks[-1][1].synchronize()
        out = {}
        for (_, a), (name, b) in zip(self.marks[:-1], self.marks[1:]):
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out


class SoloComm:
    """The collective interface of :func:`search_shards` for a single process (world size 1)."""
    world = 1

    def gather(self, t):
        return t.unsqueeze(0)

    def max_(self, t):
        return t

    def sum_int(self, v):
        return int(v)

    def sum_(self, t):
        return t


def _row_topj(vals, counts, j):
    rows, cols = vals.shape
    out = torch.empty((rows, j), dtype=torch.float32, device=vals.device)
    if rows:
        N.call("xmve_row_topj", N.ptr(vals), rows, cols, vals.stride(0), N.ptr(counts), j, N.ptr(out), N.stream_ptr())
    return out


def _row_kth(vals, counts, j1, sub, j2, sub_dev=None):
    """``max(kth(row, j1) - sub * sub_dev[0], kth(row, j2))`` per row (``sub_dev`` None: ``- sub``)."""
    rows, cols = vals.shape
    out = torch.empty((rows,), dtype=torch.float32, device=vals.device)
    if rows:
        N.call("xmve_row_kth", N.ptr(vals), rows, cols, vals.stride(0), N.ptr(counts), j1, float(sub), N.ptr(sub_dev), j2,
               N.ptr(out), N.stream_ptr())
    return out


def _eps_device(q_res, dv2, wts, n_space, k_len):
    """:func:`measured_eps` on the device: fp32 ``[1]`` tensor (no host round trip)."""
    out = torch.empty((1,), dtype=torch.float32, device=q_res.device)
    N.call("xmve_eps_bound", N.ptr(q_res), n_space, q_res.shape[1], N.ptr(dv2), math.sqrt(sum(w * w for w in wts)),
           int(k_len), eps_fallback(wts, n_space, k_len), N.ptr(out), N.stream_ptr())
    return out


def _count_before(exact, cand_idx, counts, idx_offset, s_gt, g, out):
    """``out[e] += #{candidates of entry e that precede its ground truth}`` (exact score above ``s_gt[e]``, or equal
    with a smaller global row than ``g[e]``)."""
    n_ent, cap = exact.shape
    if n_ent:
        N.call("xmve_count_before", N.ptr(exact), N.ptr(cand_idx), N.ptr(counts), n_ent, cap, int(idx_offset),
               N.ptr(s_gt), N.ptr(g), N.ptr(out), N.stream_ptr())


def _pilot_bound(lists, k, eps_t):
    """``lists`` fp64 ``[n_seg, nq, m]`` (descending per segment) -> round_down(k-th largest of the union - eps)."""
    n_seg, nq, m = lists.shape
    out = torch.empty((nq,), dtype=torch.float32, device=lists.device)
    if nq:
        N.call("xmve_pilot_bound", N.ptr(lists), n_seg, nq, m, k, 1.0, N.ptr(eps_t), N.ptr(out), N.stream_ptr())
    return out


def packed_bytes(rows, length):
    """Bytes of one packed top-k block: scores fp64 [rows, len] | rows int64 [rows, len] | overflow int32 [rows]."""
    return int(N.lib.xmve_packed_topk_bytes(int(rows), int(length)))


def packed_views(block, rows, length):
    """Typed views (scores, idx, flags) into one packed block (a uint8 tensor of :func:`packed_bytes` bytes)."""
    n = rows * length
    return (block[: n * 8].view(torch.float64).view(rows, length),
            block[n * 8: n * 16].view(torch.int64).view(rows, length),
            block[n * 16: n * 16 + rows * 4].view(torch.int32))


def _merge_packed(packed, rows, length, k, thr, eps_t, n_bad):
    """K3 on the all-gathered packed blocks ``[n_seg, seg_bytes]`` -> (scores, idx, cert, thr_next)."""
    n_seg, seg_bytes = packed.shape
    out_s = torch.empty((rows, k), dtype=torch.float64, device=packed.device)
    out_i = torch.empty((rows, k), dtype=torch.int64, device=packed.device)
    cert = torch.empty((rows,), dtype=torch.int32, device=packed.device)
    thr_next = torch.empty((rows,), dtype=torch.float32, device=packed.device)
    if rows:
        N.call("xmve_merge_topk_packed", N.ptr(packed), n_seg, seg_bytes, rows, length, None, k, N.ptr(thr), 1.0,
               N.ptr(eps_t), N.ptr(out_s), N.ptr(out_i), N.ptr(cert), N.ptr(thr_next), N.ptr(n_bad), N.stream_ptr())
    return out_s, out_i, cert, thr_next


def _union(parts, comm):
    """Per-row lists from the local shards ``[nq, m]`` -> the union over all shards of all ranks ``[nq, G*L*m]``."""
    loc = parts[0] if len(parts) == 1 else torch.cat(parts, dim=1)
    if comm.world == 1:
        return loc
    g = comm.gather(loc.contiguous())                                   # [G, nq, L*m]
    return g.permute(1, 0, 2).reshape(loc.shape[0], -1).contiguous()


def _segments(parts, comm):
    """Per-shard tensors of one shape -> ``[G * L, *shape]`` over all shards of all ranks (one collective)."""
    loc = parts[0].unsqueeze(0) if len(parts) == 1 else torch.stack(parts)
    if comm.world == 1:
        return loc
    g = comm.gather(loc)                                                # [G, L, ...]
    return g.view((-1,) + tuple(loc.shape[1:]))


#: the pilot holds at most this many exact scores per query and shard (xmve_pilot_top)
PILOT_MAX = 1000
#: ... and the union of the pilots of all shards at most this many (xmve_pilot_bound sorts it in shared memory)
PILOT_UNION_MAX = 4096
#: re-run passes select at most this many rows per launch: from 512 rows on, the selection kernels shrink their sort
#: to max(2048, 4k) entries per row (xmve_select_topk_*), which is what the rows being re-run may not have fitted
SELECT_RERUN_ROWS = 511


class PendingSearch:
    """A search whose first pass has been enqueued.  :meth:`result` waits for the count of uncertified rows (one
    int32 copied asynchronously to pinned host memory right after the merge), re-runs those rows if there are any,
    and returns ``(scores, idx)``.  Resolving a search one step late lets the host enqueue the next batch while the
    GPU still scores this one (bench.py does that); ``search_shards(defer=False)`` resolves at once."""

    def __init__(self, ctx):
        self._ctx = ctx
        self._ctx_template = None
        self._done = ctx is None
        self.scores = self.idx = None
        self.reran = False                    # True once result() had to re-run rows (scores / idx were rewritten)

    @classmethod
    def ready(cls, scores, idx):
        p = cls(None)
        p.scores, p.idx = scores, idx
        return p

    def result(self):
        if not self._done:
            if self._ctx.dev.type == "cuda":
                with torch.cuda.device(self._ctx.dev):
                    self.reran = self._ctx.resolve()
            else:
                self.reran = self._ctx.resolve()
            self._done = True
            self._ctx = None
        return self.scores, self.idx


class _Search:
    """State of one filtered search (every rank holds the same queries, thresholds and outputs)."""

    def __init__(self, stores, comm, k, k_eff, kk, wts, excl, eps_t, pl, a_op, q_raw, q_norm, nq, thr, out_s, out_i,
                 stats, ph, masks=None, n_elig=None):
        self.stores, self.comm, self.k, self.k_eff, self.kk, self.wts = stores, comm, k, k_eff, kk, wts
        self.excl, self.eps_t, self.pl = excl, eps_t, pl
        self.a_op, self.q_raw, self.q_norm, self.nq, self.thr = a_op, q_raw, q_norm, nq, thr
        self.out_s, self.out_i, self.stats, self.ph = out_s, out_i, stats, ph
        self.ref = stores[0]
        self.dev = self.ref.device
        self.live = [s for s in stores if s.n]
        self.n_shards = len(stores) * comm.world
        self.solo = self.n_shards == 1
        cap = pl["cap"]
        if not self.solo:
            cap = max(2048, min(cap, 1 << int(math.ceil(math.log2(4.0 * cap / self.n_shards)))))
        self.cap = cap
        self.n_shard_max = max(s.n for s in self.live) if self.live else 1
        self.pending = None
        # filtered search: a row with at most `cap` eligible rows in the whole corpus gets thr = -inf -- every shard's
        # list then holds all its eligible rows, and the list is complete even when it is shorter than k
        self.masks, self.n_elig = masks, n_elig
        # (a row with no eligible row at all gets thr = +inf: nothing enters its window, and its answer is empty)
        if masks is not None:
            self.thr = torch.where(n_elig == 0, torch.full_like(thr, float("inf")),
                                   torch.where(n_elig <= cap, torch.full_like(thr, float("-inf")), thr))

    # one pass over all rows (rows None) or over the rows that are re-run --------------------------------
    def run_pass(self, rows):
        ref, dev, comm, ph, k_eff, kk, eps_t = self.ref, self.dev, self.comm, self.ph, self.k_eff, self.kk, self.eps_t
        if rows is None:
            a_sub, q_sub, qn_sub, thr_sub, ex_sub, n_sub = self.a_op, self.q_raw, self.q_norm, self.thr, self.excl, self.nq
        else:
            n_sub = rows.numel()
            a_sub = torch.zeros((_round_up(n_sub, _BM), ref.k), dtype=torch.bfloat16, device=dev)
            a_sub[:n_sub] = self.a_op[rows]
            q_sub = self.q_raw[rows].contiguous()
            qn_sub = self.q_norm[:, rows].contiguous()
            thr_sub = self.thr[rows].contiguous()
            ex_sub = self.excl[rows].contiguous() if self.excl is not None else None
        cap = self.cap
        kw = {}
        if self.masks is not None:
            kw["label_mask"] = self.masks if rows is None else self.masks[rows].contiguous()
        # 3: fused score + threshold filter on every local shard
        ph.mark("alloc")
        cands = [s._filter(a_sub, n_sub, thr_sub, cap, **kw) for s in self.live]
        ph.mark("filter")
        # 4: what needs an exact score
        m = kk if self.solo else min(kk, int(math.ceil(1.5 * kk / self.n_shards)) + 10)
        if kk <= PILOT_MAX and (self.solo or self.n_shards * m <= PILOT_UNION_MAX):
            # two rounds.  One: every shard rescores its m best approximate candidates; the k-th largest exact score
            # of the union of these pilots (kth1) is a lower bound on the true k-th best.  Two: only candidates whose
            # approximate score reaches kth1 - eps can still belong to the top-k.
            firsts = [_row_kth(c[1], c[0], m, 0.0, 0) for c in cands]
            exacts = [s._rescore(q_sub, qn_sub, n_sub, self.wts, c, b1) for s, c, b1 in zip(self.live, cands, firsts)]
            pilots = [s._pilot_top(e, c, n_sub, ex_sub, m) for s, c, e in zip(self.live, cands, exacts)]
            if not pilots:
                pilots = [torch.full((n_sub, m), float("-inf"), dtype=torch.float64, device=dev)]
            bound = _pilot_bound(_segments(pilots, comm), k_eff, eps_t)
            ph.mark("pilot")
            for s, c, b1, e in zip(self.live, cands, firsts, exacts):
                s._rescore(q_sub, qn_sub, n_sub, self.wts, c, bound, b1, e)
        else:
            # very deep lists (k > 1000): one round against (kk-th largest approximate score over all shards) - 2 eps
            if self.solo:
                bound = _row_kth(cands[0][1], cands[0][0], kk, 2.0, 0, eps_t)
            elif kk <= ROW_TOPJ_MAX:
                tops = [_row_topj(c[1], c[0], kk) for c in cands]
                if not tops:
                    tops = [torch.full((n_sub, kk), float("-inf"), dtype=torch.float32, device=dev)]
                bound = _row_kth(_union(tops, comm), None, kk, 2.0, 0, eps_t)
            else:
                # deeper than xmve_row_topj extracts: the best shard's own kk-th largest approximate score is a lower
                # bound on the kk-th largest of the union (looser, so a few more rows are rescored)
                bound = torch.full((n_sub,), float("-inf"), dtype=torch.float32, device=dev)
                for c in cands:
                    bound = torch.maximum(bound, _row_kth(c[1], c[0], kk, 2.0, 0, eps_t))
                bound = comm.max_(bound)
            ph.mark("bound")
            exacts = [s._rescore(q_sub, qn_sub, n_sub, self.wts, c, bound) for s, c in zip(self.live, cands)]
        ph.mark("rescore")
        # 5: selection.  One shard: the local kernel certifies.  Several: packed local lists, ONE gather, K3.
        # With 512 rows or more the selection kernels sort at most max(2048, 4k) entries per row; a re-run selects in
        # smaller batches, so that the rows whose lists did not fit (heavy float ties) get the full 16 384 entries.
        n_bad = torch.zeros((1,), dtype=torch.int32, device=dev)
        batch = n_sub if rows is None else SELECT_RERUN_ROWS
        parts = [self._select_rows(r0, min(n_sub, r0 + batch), cands, exacts, ex_sub, thr_sub, bound, n_bad)
                 for r0 in range(0, n_sub, batch)]
        if len(parts) == 1:
            s_, i_, cert, thr_next, over = parts[0]
        else:
            s_, i_, cert, thr_next = (torch.cat([p[j] for p in parts]) for j in range(4))
            over = ("parts", [p[4] for p in parts])
        if self.masks is not None:
            # a row with thr = -inf whose lists did not overflow holds every eligible row.  When it holds fewer than k
            # (its last entry is padding) the selection cannot certify it, yet it is exact; a row with k entries or
            # more keeps the selection's verdict (which also covers float ties cut by the sort).  A row without any
            # eligible row is empty.
            n_elig = self.n_elig if rows is None else self.n_elig[rows]
            short = (thr_sub == float("-inf")) & ~self._overflowed(over) & (i_[:, -1] == -1)
            cert = torch.where(short | (n_elig == 0), torch.ones_like(cert), cert)
            n_bad.copy_((cert == 0).sum().reshape(1))
        ph.mark("select_merge")
        if self.stats is not None and rows is None:
            st = self.stats
            st["eps"] = float(eps_t)
            st["cap"] = cap
            st["pilot_m"] = m
            st["cand_count"] = [c[0] for c in cands]
            ar = torch.arange(cap, device=dev)
            st["rescored_per_query"] = sum(
                float(((ar[None, :] < c[0][:, None]) & (e[:, :cap] > float("-inf"))).sum())
                for c, e in zip(cands, exacts)) / max(n_sub, 1)
            if self.masks is not None:
                st["eligible_min"], st["eligible_max"] = int(self.n_elig.min()), int(self.n_elig.max())
                st["thr_inf_rows"] = int((thr_sub == float("-inf")).sum())
            ph.mark("stats_bookkeeping")
        return s_, i_, cert, thr_next, over, n_bad, thr_sub

    def _select_rows(self, r0, r1, cands, exacts, ex_sub, thr_sub, bound, n_bad):
        """Step 5 for rows ``r0:r1`` of a pass -> (scores, idx, cert, thr_next, overflow descriptor)."""
        dev, k_eff, eps_t, cap = self.dev, self.k_eff, self.eps_t, self.cap
        n = r1 - r0
        cands = [tuple(t[r0:r1] for t in c) for c in cands]
        exacts = [e[r0:r1] for e in exacts]
        ex = ex_sub[r0:r1] if ex_sub is not None else None
        thr = thr_sub[r0:r1]
        if self.solo:
            s_ = torch.empty((n, k_eff), dtype=torch.float64, device=dev)
            i_ = torch.empty((n, k_eff), dtype=torch.int64, device=dev)
            cert, thr_next = self.live[0]._select(exacts[0], cands[0], n, k_eff, ex, thr, eps_t, bound[r0:r1], s_, i_,
                                                  True, n_bad)
            return s_, i_, cert, thr_next, ("lists", [cands[0][0]], cap)
        seg = packed_bytes(n, k_eff)
        blocks = torch.empty((max(len(self.live), 1), seg), dtype=torch.uint8, device=dev)
        for li, (s, c, e) in enumerate(zip(self.live, cands, exacts)):
            b_s, b_i, b_f = packed_views(blocks[li], n, k_eff)
            exact_list, _ = s._select(e, c, n, k_eff, ex, None, eps_t, None, b_s, b_i, False)
            b_f.copy_(exact_list == 0)                        # overflowed, or cut short by float ties
        if not self.live:
            b_s, b_i, b_f = packed_views(blocks[0], n, k_eff)
            b_s.fill_(float("-inf"))
            b_i.fill_(-1)
            b_f.zero_()
        gathered = blocks if self.comm.world == 1 else self.comm.gather(blocks).view(-1, seg)
        s_, i_, cert, thr_next = _merge_packed(gathered, n, k_eff, k_eff, thr, eps_t, n_bad)
        return s_, i_, cert, thr_next, ("packed", gathered, n, k_eff)

    def first_pass(self, in_graph=False, flag_host=None):
        self._cap0 = self.cap
        s_, i_, cert, thr_next, over, n_bad, thr_sub = self.run_pass(None)
        self.out_s[:, :self.k_eff] = s_
        self.out_i[:, :self.k_eff] = i_
        self._last = (cert, thr_next, over, thr_sub)
        if self.dev.type == "cuda":
            # (pinned memory is allocated outside a graph capture: GraphSearch passes its own buffer)
            self._flag = torch.empty((1,), dtype=torch.int32).pin_memory() if flag_host is None else flag_host
            self._flag.copy_(n_bad, non_blocking=True)
            self._event = None
            if not in_graph:                                  # a captured event cannot be waited on: see replayed()
                self._event = torch.cuda.Event()
                self._event.record()
        else:
            self._flag, self._event = n_bad, None
        self._thr0 = self.thr

    def replayed(self):
        """The captured first pass has just been replayed (GraphSearch): mark the point the host waits for."""
        self.thr = self._thr0                                 # a re-run of the previous batch may have replaced it
        self.cap = self._cap0                                 # ... or grown the candidate lists
        self._event = torch.cuda.Event()
        self._event.record()

    def resolve(self):
        """Wait for the first pass's certificate count; re-run (all ranks alike) the rows that missed it."""
        if self._event is not None:
            self._event.synchronize()
        self.ph.mark("certify_sync")
        reran = int(self._flag[0]) != 0
        if reran:
            self._rerun()
        if self.stats is not None:
            self.stats["phases_ms"] = self.ph.result()
        return reran

    @staticmethod
    def _overflowed(over):
        """Per-row overflow flags of a pass (formed only when rows are re-run)."""
        if over[0] == "parts":
            return torch.cat([_Search._overflowed(o) for o in over[1]])
        if over[0] == "lists":
            return over[1][0] > over[2]
        _, gathered, n_sub, k_eff = over
        flags = torch.stack([packed_views(gathered[g], n_sub, k_eff)[2] for g in range(gathered.shape[0])])
        return flags.max(dim=0).values != 0

    def _rerun(self):
        cert, thr_next, over, thr_sub = self._last
        rows = None
        for attempt in range(12):
            bad = torch.nonzero(cert == 0).flatten()            # device -> host sync (identical on every rank)
            if bad.numel() == 0:
                return
            over = self._overflowed(over)
            # an overflowed row needs a HIGHER threshold; if the kernel cannot propose one, grow the lists
            stuck = over[bad] & (thr_next[bad] <= thr_sub[bad])
            if rows is None:
                self.thr = self.thr.clone()
                self.thr[bad] = thr_next[bad]
                rows = bad
            else:
                self.thr[rows[bad]] = thr_next[bad]
                rows = rows[bad]
            if self.stats is not None:
                self.stats["reruns"] = self.stats.get("reruns", 0) + 1
                self.stats["rerun_rows"] = self.stats.get("rerun_rows", 0) + int(rows.numel())
            if bool(stuck.any()):
                # overflow that a tighter threshold cannot fix (dense neighbourhoods within eps of the k-th best):
                # grow the lists -- for the few rows left they may grow until they hold a whole shard
                room = max(32768, min(1 << int(math.ceil(math.log2(self.n_shard_max))),
                                      (1 << 27) // max(int(rows.numel()), 1)))
                self.cap = min(room, self.cap * 4)
            if self.masks is not None:                        # rows whose eligible rows now fit the lists
                self.thr[rows] = torch.where(self.n_elig[rows] <= self.cap,
                                             torch.full_like(self.thr[rows], float("-inf")), self.thr[rows])
            s_, i_, cert, thr_next, over, _, thr_sub = self.run_pass(rows)
            self.out_s[rows, :self.k_eff] = s_
            self.out_i[rows, :self.k_eff] = i_
        bad = torch.nonzero(cert == 0).flatten()
        if bad.numel():
            raise N.XmveError("search: %d row(s) could not be certified after 12 passes (increase eps headroom "
                              "or candidate capacity; heavy score ties?)" % int(bad.numel()))


class GraphSearch:
    """A search of fixed shape captured ONCE into a CUDA graph and replayed per query batch.

    The first pass of :func:`search_shards` never waits for the host and has static shapes for a given
    ``(number of queries, k, weights, exclude yes/no)``: about 25 kernel launches and as many small allocations, which
    cost the host ~0.4 ms -- more than the GPU needs for a handful of queries (online search, the 60-query AVS batch).
    Replaying the captured graph costs ~10 us of host time.  The rare uncertified rows are re-run eagerly by
    :meth:`PendingSearch.result`, exactly as without a graph.

        gs = GraphSearch(store, n_queries=60, k=1000)
        scores, idx = gs(queries)                 # or  p = gs(queries, defer=True); ...; p.result()

    With ``comm`` (``distributed.GroupComm``) the NCCL gathers of a sharded search are captured inside the graph and
    every rank replays in lockstep (``tools/check_sharded.py`` / ``tools/graph_sharded_check.py``: identical to the
    eager search; 0.94 -> 0.64 ms for 60 queries over two 135 k-row shards, where the ~40 launches of the eager step
    are what bounds it).  The returned tensors are the graph's static output buffers and are overwritten by the
    next call.  The graph covers the rows the stores held at capture: a call after :meth:`CorpusStore.add` raises.

    ``with_label_mask=True`` captures a filtered search: ``gs(queries, label_mask=...)`` (one mask per query or one
    for all; None = every label).  The graph also covers the labels held at capture: a call after
    :meth:`CorpusStore.set_labels` raises.
    """

    def __init__(self, stores, n_queries, k, weights=None, with_exclude=False, comm=None, n_total=None,
                 small_nv=SMALL_NV, with_label_mask=False):
        self.stores = list(stores) if isinstance(stores, (list, tuple)) else [stores]
        ref = self.stores[0]
        self.dev = ref.device
        self.nq, self.k = int(n_queries), int(k)
        self.comm = comm or SoloComm()
        self.q_in = torch.randn((self.nq, ref.dtot), dtype=torch.float32, device=self.dev)   # warm-up queries
        self.excl_in = torch.full((self.nq,), -1, dtype=torch.int64, device=self.dev) if with_exclude else None
        self.mask_in = torch.full((self.nq,), -1, dtype=torch.int64, device=self.dev) if with_label_mask else None
        kw = dict(weights=weights, exclude=self.excl_in, eps=None, small_nv=small_nv, stats=None, comm=self.comm,
                  n_total=n_total)
        with torch.cuda.device(self.dev):
            # warm-up outside the capture: opt-in shared-memory attributes, the cached corpus residual, NCCL
            torch.cuda.synchronize()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    _search_shards(self.stores, self.q_in, self.k, kw["weights"], kw["exclude"], None, small_nv, None,
                                   self.comm, n_total, label_mask=self.mask_in).result()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._flag_host = torch.empty((1,), dtype=torch.int32).pin_memory()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._pending = _search_shards(self.stores, self.q_in, self.k, kw["weights"], kw["exclude"], None,
                                               small_nv, None, self.comm, n_total, in_graph=True,
                                               flag_host=self._flag_host, label_mask=self.mask_in)
        self.scores, self.idx = self._pending.scores, self._pending.idx
        self.rows = tuple(s.n for s in self.stores)           # the captured kernels cover exactly these rows
        self.label_versions = tuple(s.label_version for s in self.stores)   # ... and, filtered, these labels

    def __call__(self, queries, exclude=None, defer=False, label_mask=None):
        q = queries if torch.is_tensor(queries) else torch.as_tensor(queries)
        assert tuple(q.shape) == tuple(self.q_in.shape), "GraphSearch was captured for %s queries" % (self.q_in.shape,)
        rows = tuple(s.n for s in self.stores)
        if rows != self.rows:
            raise RuntimeError("GraphSearch: the corpus changed since the capture (rows per store %s, now %s); the "
                               "captured kernels would not see the new rows -- capture a new GraphSearch"
                               % (list(self.rows), list(rows)))
        if self.mask_in is not None and tuple(s.label_version for s in self.stores) != self.label_versions:
            raise RuntimeError("GraphSearch: set_labels ran since the capture; the captured eligible-row counts are "
                               "stale -- capture a new GraphSearch")
        with torch.cuda.device(self.dev):
            self.q_in.copy_(q, non_blocking=True)
            if self.excl_in is not None:
                e = torch.full((self.nq,), -1, dtype=torch.int64) if exclude is None else torch.as_tensor(exclude)
                self.excl_in.copy_(e.to(torch.int64), non_blocking=True)
            else:
                assert exclude is None, "capture with with_exclude=True to pass exclusions"
            if self.mask_in is not None:
                self.mask_in.copy_(_label_masks(-1 if label_mask is None else label_mask, self.nq, self.dev))
            elif label_mask is not None:
                raise ValueError("capture with with_label_mask=True to pass label masks")
            self.graph.replay()
            ctx = self._pending._ctx_template
            ctx.replayed()
            p = PendingSearch(ctx)
            p.scores, p.idx = self.scores, self.idx
        return p if defer else p.result()


def _eps_for(stores, comm, wts, eps, q_res):
    """The error bound as a device fp32 ``[1]``: measured (:func:`_eps_device`), or the caller's ``eps`` per unit of
    fusion weight."""
    ref = stores[0]
    if eps is None:
        return _eps_device(q_res, _dv2_global(stores, comm), wts, len(ref.dims), ref.k)
    return torch.full((1,), float(eps) * max(1.0, sum(abs(w) for w in wts)), dtype=torch.float32, device=ref.device)


def _dv2_global(stores, comm):
    """max over ALL corpus rows (every shard of every rank) of the squared bf16 residual: device fp32 [1], cached per
    corpus state -- the one all-reduce it needs is paid when the corpus changes, not per search."""
    ref = stores[0]
    key = (tuple(s.n for s in stores), comm.world)
    cached = getattr(ref, "_dv2_cache", None)
    if cached is not None and cached[0] == key:
        return cached[1]
    v = torch.stack([s.resid_max2().reshape(()) for s in stores]).max().reshape(1).float()
    v = comm.max_(v)
    ref._dv2_cache = (key, v)
    return v


def _label_hist_global(stores, comm):
    """Label histogram over ALL corpus rows (every shard of every rank): device int64 [64], cached per corpus and
    label state like :func:`_dv2_global` -- the all-reduce is paid when rows or labels change, not per search."""
    ref = stores[0]
    key = (tuple((s.n, s.label_version) for s in stores), comm.world)
    cached = getattr(ref, "_label_hist_cache", None)
    if cached is not None and cached[0] == key:
        return cached[1]
    h = comm.sum_(torch.stack([s._label_counts() for s in stores]).sum(0))
    ref._label_hist_cache = (key, h)
    return h


def search_shards(stores, queries, k, weights=None, exclude=None, eps=None, small_nv=SMALL_NV, stats=None, comm=None,
                  n_total=None, defer=False, head_stream=None, label_mask=None):
    """Exact top-``k`` over a corpus cut into shards: ``stores`` are this process's shards (normally one), ``comm``
    joins the processes of a ``torch.distributed`` group (``distributed.GroupComm``; every rank calls this function
    with the same queries).  All shards work against ONE per-query threshold:

    1. K1 on the query batch; the measured error bound ``eps`` as a device scalar (the corpus-side maximum is
       all-reduced once per corpus state, the query side is identical on every rank).
    2. the largest scores of a ``step``-strided sample of each shard (a coarse K2 STORE pass sets a floor, a K2
       FILTER pass over the sample keeps what exceeds it); the top-J of every shard are gathered and the global
       threshold is ``max(kth(union, j) - thr_margin(k / step) * eps, kth(union, j_cap))`` -- what one GPU would compute on the whole
       corpus, so each shard appends only its share of the candidates.
    3. K2 FILTER over each shard (the score matrix never reaches HBM).
    4. exact fp64 rescore in two rounds: every shard rescores its best ``m`` approximate candidates; the pilots are
       gathered and the k-th largest exact score of their union, minus eps, bounds what the second round rescores
       (about half of what the one-round window ``approximate k-th - 2 eps`` needs).
    5. local top-k per shard into a packed block; ONE gather of the blocks; merge (K3) with the certificate
       ``kth_exact - eps >= threshold`` and no overflowed list.
    6. rows without a certificate are re-run (by all ranks alike) with the threshold the merge proposes.  Their
       number is the only thing the host reads back, asynchronously: with ``defer=True`` the function returns a
       :class:`PendingSearch` right after enqueueing steps 1-5 and ``.result()`` does step 6.

    Corpora of at most ``small_nv`` rows skip 2-4: every shard forms its fp64 score matrix directly.
    With one shard and one rank no gather happens and the certificate comes from the local selection kernel.

    ``head_stream`` (a ``torch.cuda.Stream``; use with ``defer=True``): steps 1-2 are enqueued on that stream and the
    current stream only waits for their result before step 3.  Batches are independent, so when the caller keeps one
    search in flight the K1 / sampling / threshold work of batch i+1 runs next to the rescore / selection / merge of
    batch i as soon as FILTER(i) has left the SMs, instead of behind it -- both are short, latency-bound kernel
    chains (1.2 ms + 1.9 ms of a 31 ms step on 8 GPUs).  The queries must be complete when the call is made, or have
    been produced on ``head_stream`` (it does not wait for the current stream).  The head does wait for the last
    :meth:`CorpusStore.add` of every store it reads (an event recorded by ``add``), so a search issued straight after
    an ``add`` sees the new rows and their residuals.

    ``label_mask`` restricts each query to the rows whose label its mask allows (:meth:`CorpusStore.search`).  The
    samples and the FILTER see eligible rows only; a query with at most ``cap`` eligible rows gets thr = -inf, so its
    lists are complete and certified however short.  ``None`` runs the unfiltered pipeline unchanged.
    """
    comm = comm or SoloComm()
    ref = stores[0]
    if ref.device.type == "cuda":
        with torch.cuda.device(ref.device):                     # kernels, streams and allocations follow the store
            pending = _search_shards(stores, queries, k, weights, exclude, eps, small_nv, stats, comm, n_total,
                                     head_stream=head_stream, label_mask=label_mask)
            return pending if defer else pending.result()
    pending = _search_shards(stores, queries, k, weights, exclude, eps, small_nv, stats, comm, n_total,
                             label_mask=label_mask)
    return pending if defer else pending.result()


def _head_on(stream):
    import contextlib
    return torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()


def _search_shards(stores, queries, k, weights, exclude, eps, small_nv, stats, comm, n_total, in_graph=False,
                   flag_host=None, head_stream=None, label_mask=None):
    ref = stores[0]
    dev, n_space = ref.device, len(ref.dims)
    n_shards = len(stores) * comm.world
    solo = n_shards == 1
    n_local = sum(s.n for s in stores)
    if n_total is None:
        n_total = comm.sum_int(n_local)
    if n_total == 0:
        raise ValueError("empty corpus")
    wts = _weights(weights, n_space)
    ph = _Phases(stats is not None and ref.device.type == "cuda")
    ph.mark("start")
    nq_in = (queries[0] if isinstance(queries, (list, tuple)) else queries).shape[0]
    # the head (steps 1-2) on its own stream: filtered searches only, and not while phases are being timed
    if dev.type != "cuda" or stats is not None or in_graph or n_total <= small_nv or nq_in == 0:
        head_stream = None
    if head_stream is not None:
        for t in (queries if isinstance(queries, (list, tuple)) else (queries, exclude)):
            if torch.is_tensor(t) and t.is_cuda:
                t.record_stream(head_stream)                  # the caller may drop it while the head still reads it
        if torch.is_tensor(label_mask) and label_mask.is_cuda:
            label_mask.record_stream(head_stream)
        for s in stores:                                      # the head reads the stores' rows and residuals: only
            if getattr(s, "added", None) is not None:         # their last add, not the whole current stream, must
                head_stream.wait_event(s.added)               # be complete
    with _head_on(head_stream):
        a_op, q_raw, q_norm, q_res, nq = ref.prepare_queries(queries, wts)
        excl = None
        if exclude is not None:
            excl = torch.as_tensor(exclude, dtype=torch.int64).to(dev).contiguous()   # the kernels read excl[q]
        masks = n_elig = None
        if label_mask is not None:
            masks = _label_masks(label_mask, nq, dev)
            n_elig = _eligible_counts(masks, _label_hist_global(stores, comm))
    ph.mark("prepare_queries")
    if nq == 0:
        return PendingSearch.ready(torch.empty((0, k), dtype=torch.float64, device=dev),
                                   torch.empty((0, k), dtype=torch.int64, device=dev))
    k_eff = min(int(k), n_total)
    out_s = torch.full((nq, k), float("-inf"), dtype=torch.float64, device=dev)
    out_i = torch.full((nq, k), -1, dtype=torch.int64, device=dev)

    if n_total <= small_nv:
        kw = {} if masks is None else {"label_mask": masks}
        parts = [s._exact_small(q_raw, q_norm, nq, k_eff, wts, excl, **kw) for s in stores if s.n]
        if not parts:
            parts = [(torch.full((nq, k_eff), float("-inf"), dtype=torch.float64, device=dev),
                      torch.full((nq, k_eff), -1, dtype=torch.int64, device=dev))]
        if solo:
            s_, i_ = parts[0]
        else:
            s_, i_ = _merge(_union([p[0] for p in parts], comm), _union([p[1] for p in parts], comm), k_eff)
        out_s[:, :k_eff] = s_
        out_i[:, :k_eff] = i_
        return PendingSearch.ready(out_s, out_i)

    kk = k_eff + (1 if excl is not None else 0)               # one extra in case the excluded row is among them
    pl = plan(kk, n_total)
    with _head_on(head_stream):
        eps_t, thr = _threshold(stores, comm, solo, wts, eps, pl, a_op, q_res, nq, ph, masks)
    if head_stream is not None:
        # step 3 onwards runs on the caller's stream: it waits for the head, and the caching allocator must not hand
        # the head's tensors back to the head stream while this stream still reads them
        main = torch.cuda.current_stream()
        main.wait_stream(head_stream)
        for t in (a_op, q_raw, q_norm, q_res, eps_t, thr, excl, masks, n_elig):
            if t is not None:
                t.record_stream(main)
    search = _Search(stores, comm, k, k_eff, kk, wts, excl, eps_t, pl, a_op, q_raw, q_norm, nq, thr, out_s, out_i,
                     stats, ph, masks, n_elig)
    search.first_pass(in_graph, flag_host)
    pending = PendingSearch(search)
    pending._ctx_template = search
    pending.scores, pending.idx = out_s, out_i
    return pending


def _threshold(stores, comm, solo, wts, eps, pl, a_op, q_res, nq, ph, masks=None):
    """Steps 1b-2 of :func:`search_shards`: the error bound and the per-query threshold -> (eps_t, thr).  With
    ``masks`` the samples hold eligible rows only: the strided sample keeps its meaning among them (about k / step
    of a query's top-k eligible rows are sampled), so :func:`plan` applies unchanged."""
    dev = stores[0].device
    eps_t = _eps_for(stores, comm, wts, eps, q_res)
    ph.mark("eps")
    live = [s for s in stores if s.n]
    # 2: one global threshold from the shards' samples
    j_cap = pl["j_cap"] if solo else min(pl["j_cap"], ROW_TOPJ_MAX)      # xmve_row_topj holds 4096 values per row
    big_j = max(pl["j"], j_cap)
    kw = {} if masks is None else {"label_mask": masks}
    lists, floor = [], torch.full((nq,), float("-inf"), dtype=torch.float32, device=dev)
    for s in live:
        if (s.n + pl["step"] - 1) // pl["step"] >= 16384:
            # two-level: the sample matrix (2.1 GB at 10 M rows) is never written or radix-selected
            sc, cnt, thr0 = s._sample_top(a_op, nq, pl["step"], big_j, **kw)
            lists.append((sc, cnt))
            floor = thr0 if len(lists) == 1 else torch.minimum(floor, thr0)
        else:                                                 # small shard: the few launches of the plain way win
            lists.append((s._sample(a_op, nq, pl["step"], **kw), None))
            floor = torch.full_like(floor, float("-inf"))     # a complete list needs no floor
    if solo:
        thr = _row_kth(lists[0][0], lists[0][1], pl["j"], pl["margin"], j_cap, eps_t)
    elif big_j > ROW_TOPJ_MAX:
        # more order statistics than xmve_row_topj extracts (k in the thousands over a small corpus): the j-th largest
        # of ONE shard's sample is a lower bound on the j-th largest of the union -- a valid, lower threshold; lists
        # that overflow because of it go through the re-run path
        thr = torch.full((nq,), float("-inf"), dtype=torch.float32, device=dev)
        for sc, cnt in lists:
            thr = torch.maximum(thr, _row_kth(sc, cnt, pl["j"], pl["margin"], 0, eps_t))
        thr = comm.max_(thr)
        floor = -comm.max_(-floor)
    else:
        tops = [_row_topj(sc, cnt, big_j) for sc, cnt in lists]
        if not tops:
            tops = [torch.full((nq, big_j), float("-inf"), dtype=torch.float32, device=dev)]
        tops.append(floor.unsqueeze(1))                       # the floors ride along with the order statistics
        u = _union(tops, comm)                                # [nq, G * (L * big_j + 1)]
        per = u.shape[1] // comm.world
        floor = u.view(nq, comm.world, per)[:, :, -1].min(dim=1).values
        u.view(nq, comm.world, per)[:, :, -1] = float("-inf")
        thr = _row_kth(u, None, pl["j"], pl["margin"], j_cap, eps_t)
    # a two-level list that came out too short gives -inf (or a value below the floor): fall back to the coarse
    # floor, which ~0.4 % of the corpus exceeds -- far more than k rows, so it is below the k-th best score
    thr = torch.maximum(thr, floor - 2.0 * eps_t)
    del lists
    ph.mark("sample_threshold")
    return eps_t, thr


def rank_of_gt(stores, queries, gt_off, gt_rows, weights=None, comm=None, n_total=None, cap=8192, eps=None,
               stats=None, label_mask=None):
    """EXACT rank of every ground-truth item when the score matrix cannot exist (C3-C5 scale), sharded.

    ``gt_off`` int64 ``[nq + 1]`` / ``gt_rows`` int64 ``[E]`` are a CSR of global corpus rows per query (host arrays
    or tensors).  Returns ``ranks`` int32 ``[E]`` on the device: ``1 + #{v : s(v) > s(g)} + #{v < g : s(v) == s(g)}``
    with ``s`` the exact fp64 fused score -- the position of ``g`` in the stable ascending argsort of the reference's
    errors row (``util/metrics.py:139-145``).  Feed them to ``metrics.RankResult.from_ranks`` for R@K / MedR / MeanR /
    mAP.

    1. the shard that owns ``g`` computes ``s(g)`` with the rescore kernel; one all-reduce(max) shares it.
    2. the tensor-core FILTER runs with one operand row per ENTRY and the window ``(s(g) - eps, s(g) + eps]``:
       rows above the window are counted (they are certainly better: ``|approx - exact| <= eps``), rows inside it
       are listed, rescored exactly and compared with ``s(g)`` (``xmve_count_before``); rows below are certainly
       worse.  Shards add their counts with ONE all-reduce(sum).
    3. entries whose window holds more than ``cap`` rows (ground truths ranked tens of thousands deep) fall back to
       an exact fp64 pass over the corpus (chunked ``xmve_score_f64`` + ``xmve_count_band_f64``).

    Ranks are over the whole corpus: ``label_mask`` is refused (ValueError).
    """
    if label_mask is not None:
        raise ValueError("rank_of_gt: ranks among label-filtered rows are not supported; label_mask must be None")
    comm = comm or SoloComm()
    stores = list(stores) if isinstance(stores, (list, tuple)) else [stores]
    ref = stores[0]
    dev, n_space = ref.device, len(ref.dims)
    wts = _weights(weights, n_space)
    if n_total is None:
        n_total = comm.sum_int(sum(s.n for s in stores))
    import contextlib
    with (torch.cuda.device(dev) if dev.type == "cuda" else contextlib.nullcontext()):
        a_op, q_raw, q_norm, q_res, nq = ref.prepare_queries(queries, wts)
        off = torch.as_tensor(gt_off, dtype=torch.int64)
        g = torch.as_tensor(gt_rows, dtype=torch.int64).to(dev)
        n_ent = int(g.numel())
        assert off.numel() == nq + 1 and int(off[-1]) == n_ent, "gt_off must be a CSR over the query rows"
        if n_ent == 0:
            return torch.zeros((0,), dtype=torch.int32, device=dev)
        owner = torch.repeat_interleave(torch.arange(nq), off[1:] - off[:-1]).to(dev)        # entry -> query row
        eps_t = _eps_for(stores, comm, wts, eps, q_res)
        # one operand / raw row per entry
        a_ent = torch.zeros((_round_up(n_ent, _BM), ref.k), dtype=torch.bfloat16, device=dev)
        a_ent[:n_ent] = a_op[owner]
        q_ent = q_raw[owner].contiguous()
        qn_ent = q_norm[:, owner].contiguous()
        live = [s for s in stores if s.n]
        # 1: exact score of every ground-truth item, from the shard that owns it
        s_gt = comm.max_(_row_scores(live, q_ent, qn_ent, n_ent, wts, g))
        if bool((s_gt == float("-inf")).any()):
            raise IndexError("rank_of_gt: a ground-truth row is outside the corpus (or its score is not finite)")
        # 2-3: rows before g
        before, n_deep = _count_before_all(live, comm, a_ent, q_ent, qn_ent, n_ent, wts, s_gt, g, eps_t, cap)
        if stats is not None:
            stats["eps"] = float(eps_t)
            stats["deep_entries"] = n_deep
        return (before + 1).to(torch.int32)


def _row_scores(live, q_ent, qn_ent, n_ent, wts, g, masks=None):
    """Exact fp64 score of global row ``g[e]`` for entry ``e``, from the local shard that owns it; -inf where no local
    shard owns ``g[e]`` (or, with ``masks``, where its label is not allowed).  The caller all-reduces (max) over
    ranks."""
    dev = q_ent.device
    s_gt = torch.full((n_ent,), float("-inf"), dtype=torch.float64, device=dev)
    for s in live:
        mine = (g >= s.index_offset) & (g < s.index_offset + s.n)
        loc = torch.where(mine, g - s.index_offset, torch.zeros_like(g)).to(torch.int32).unsqueeze(1).contiguous()
        cnt = mine.to(torch.int32)
        ex = s._rescore(q_ent, qn_ent, n_ent, wts, (cnt, torch.zeros((n_ent, 1), device=dev), loc), None)
        if masks is not None:
            lab = s._ensure_labels()[loc[:, 0].long()].long()
            mine = mine & (torch.bitwise_and(torch.bitwise_right_shift(masks, lab), 1) != 0)
        s_gt = torch.where(mine, ex[:, 0], s_gt)
    return s_gt


def _count_before_all(live, comm, a_ent, q_ent, qn_ent, n_ent, wts, s_gt, g, eps_t, cap, masks=None):
    """Steps 2-3 of :func:`rank_of_gt`: int64 ``[n_ent]`` = #{corpus rows v of every shard of every rank (eligible
    under ``masks``) : s(v) > s_gt[e], or s(v) == s_gt[e] and v < g[e]} -> (counts, entries settled by the fp64
    fallback).  With ``g = INT64_MAX`` that is #{v : s(v) >= s_gt[e]}."""
    dev = q_ent.device
    # 2: window around s(g), widened by the float roundings of its ends
    e64 = eps_t.double()
    lo = (s_gt - 1.001 * e64 - 1e-7).float()
    hi = (s_gt + 1.001 * e64 + 1e-7).float()
    kw = {} if masks is None else {"label_mask": masks}
    tally = torch.zeros((2, n_ent), dtype=torch.int64, device=dev)                            # [before, overflowed]
    for s in live:
        above, count, c_s, c_i = s._filter_band(a_ent, n_ent, lo, hi, cap, **kw)
        ex = s._rescore(q_ent, qn_ent, n_ent, wts, (count, c_s, c_i), None)
        tally[0] += above
        _count_before(ex, c_i, count, s.index_offset, s_gt, g, tally[0])
        tally[1] += (count > cap)
        del ex, c_s, c_i
    tally = comm.sum_(tally)
    deep = torch.nonzero(tally[1] != 0).flatten()                                             # host sync
    # 3: exact fp64 pass for the entries whose window overflowed
    if deep.numel():
        kw = {} if masks is None else {"masks": masks[deep].contiguous()}
        fix = _rank_deep(live, q_ent[deep].contiguous(), qn_ent[:, deep].contiguous(), s_gt[deep].contiguous(),
                         g[deep].contiguous(), wts, **kw)
        tally[0, deep] = comm.sum_(fix)
    return tally[0], int(deep.numel())


def _rank_deep(live, q_ent, qn_ent, s_gt, g, wts, chunk=1 << 17, band_cap=64, delta=1e-13, masks=None):
    """#{rows before the ground truth} over this rank's shards from an exact fp64 score matrix, chunk by chunk.
    Scores more than ``delta`` above ``s_gt`` are counted; the handful within ``delta`` (the fp64 matrix and the
    rescore kernel sum in different orders, ~1e-15 apart) are settled by the rescore kernel itself.  ``masks``
    (int64 ``[n_ent]``): ineligible rows are set to -inf first."""
    dev = q_ent.device
    n_ent = q_ent.shape[0]
    before = torch.zeros((n_ent,), dtype=torch.int64, device=dev)
    st = N.stream_ptr()
    for s in live:
        for e0 in range(0, n_ent, 4096):
            e1 = min(n_ent, e0 + 4096)
            ne = e1 - e0
            qs_n, o = [], 0
            for d in s.dims:
                qn = torch.empty((ne, d), dtype=torch.float64, device=dev)
                src = q_ent[e0:e1, o:o + d]
                N.call("xmve_normalize_f64", N.ptr(src), N.F32, ne, d, q_ent.stride(0), N.ptr(qn), d, s.norm_mode, st)
                qs_n.append(qn)
                o += d
            for r0 in range(0, s.n, chunk):
                r1 = min(s.n, r0 + chunk)
                acc, o = None, 0
                for si, d in enumerate(s.dims):
                    vn = torch.empty((r1 - r0, d), dtype=torch.float64, device=dev)
                    vs = s.raw[r0:r1, o:o + d]
                    N.call("xmve_normalize_f64", N.ptr(vs), N.F32, r1 - r0, d, s.raw.stride(0), N.ptr(vn), d,
                           s.norm_mode, st)
                    sc = torch.empty((ne, r1 - r0), dtype=torch.float64, device=dev)
                    N.call("xmve_score_f64", N.ptr(qs_n[si]), ne, d, N.ptr(vn), r1 - r0, d, d, float(wts[si]),
                           N.ptr(sc), r1 - r0, st)
                    acc = sc if acc is None else acc.add_(sc)
                    o += d
                if masks is not None:
                    N.call("xmve_mask_scores", N.ptr(acc), N.F64, ne, r1 - r0, acc.stride(0),
                           N.ptr(s._ensure_labels()[r0:]), 1, N.ptr(masks[e0:e1]), st)
                # band_count keeps counting past the capacity: a band that did not fit (many rows tied to 1e-13, e.g.
                # exact duplicates) is listed again with room for all of it
                cap_b, above = band_cap, torch.zeros((ne,), dtype=torch.int64, device=dev)
                while True:
                    bcount = torch.zeros((ne,), dtype=torch.int32, device=dev)
                    bidx = torch.zeros((ne, cap_b), dtype=torch.int32, device=dev)
                    N.call("xmve_count_band_f64", N.ptr(acc), ne, r1 - r0, r1 - r0, r0, N.ptr(s_gt[e0:]),
                           float(delta), N.ptr(above), N.ptr(bcount), N.ptr(bidx), cap_b, st)
                    longest = int(bcount.max())
                    if longest <= cap_b:
                        break
                    cap_b = _pow2(longest)
                    above.zero_()
                before[e0:e1] += above
                bidx += r0                                                                    # shard-local rows
                ex = s._rescore(q_ent[e0:e1], qn_ent[:, e0:e1].contiguous(), ne, wts,
                                (bcount, torch.zeros((ne, cap_b), device=dev), bidx), None)
                _count_before(ex, bidx, bcount, s.index_offset, s_gt[e0:e1], g[e0:e1], before[e0:e1])
                del acc, ex
    return before


#: range search: candidate lists of the first FILTER pass; longer lists are sized from the exact counts and re-run
RANGE_CAP0 = 2048
#: ... in passes of at most this many list entries (rows x cap), as the top-k re-run bounds its lists
RANGE_PASS_ENTRIES = 1 << 27
#: ... and at most this many re-run passes (the counts are exact, so one suffices unless the FILTER disagrees with
#: itself)
RANGE_PASSES = 4
#: xmve_range_select sorts rows of up to this many matches in shared memory, longer ones in a scratch buffer
RANGE_SMEM_MAX = 16384


class RangeResult:
    """The lists of a range search as a CSR on the device: query ``q``'s rows are ``idx[offsets[q]:offsets[q + 1]]``
    (int64 global rows) with their exact scores ``scores[...]`` (fp64), sorted by (score desc, row asc).
    ``offsets`` is int64 ``[nq + 1]``."""

    def __init__(self, offsets, scores, idx):
        self.offsets, self.scores, self.idx = offsets, scores, idx

    def padded(self):
        """``(scores fp64 [nq, max_count], idx int64 [nq, max_count])``, padded with -inf / -1: the layout of
        :meth:`CorpusStore.search` (``avs.write_run_file``, the CLI)."""
        nq = self.offsets.numel() - 1
        lens = self.offsets[1:] - self.offsets[:-1]
        width = int(lens.max()) if nq else 0
        dev = self.offsets.device
        out_s = torch.full((nq, width), float("-inf"), dtype=torch.float64, device=dev)
        out_i = torch.full((nq, width), -1, dtype=torch.int64, device=dev)
        if self.idx.numel():
            row = torch.repeat_interleave(torch.arange(nq, device=dev), lens)
            col = torch.arange(self.idx.numel(), device=dev) - self.offsets[row]
            out_s[row, col] = self.scores
            out_i[row, col] = self.idx
        return out_s, out_i

    def pairs(self):
        """COO form in CSR order: ``(row int64, idx int64, scores fp64)`` on the device, ``row[e]`` the list (query,
        or stored row of :meth:`CorpusStore.similar_pairs`) that entry ``e`` belongs to."""
        n = self.offsets.numel() - 1
        row = torch.repeat_interleave(torch.arange(n, device=self.offsets.device), self.offsets[1:] - self.offsets[:-1])
        return row, self.idx, self.scores


def _min_scores(min_score, nq, device):
    """``min_score`` (a float or one per query) -> fp64 device tensor ``[nq]``; ValueError on NaN or a wrong shape."""
    if torch.is_tensor(min_score):
        m = min_score.detach().to("cpu", torch.float64)
    else:
        import numpy as np
        m = torch.from_numpy(np.array(min_score, dtype=np.float64))
    if m.dim() == 0 or m.numel() == 1:
        m = m.reshape(1).expand(nq)
    if tuple(m.shape) != (nq,):
        raise ValueError("min_score: expected one value per query (%d) or one for all, got shape %s"
                         % (nq, tuple(m.shape)))
    if bool(torch.isnan(m).any()):
        raise ValueError("min_score: NaN")
    return m.contiguous().to(device)


def _range_setup(stores, queries, min_score, weights, exclude, label_mask, eps, comm):
    """K1 on the queries, the per-query minimum, exclusions, label masks and the error bound of a range call."""
    ref = stores[0]
    dev = ref.device
    wts = _weights(weights, len(ref.dims))
    a_op, q_raw, q_norm, q_res, nq = ref.prepare_queries(queries, wts)
    ms = _min_scores(min_score, nq, dev)
    excl = None
    if exclude is not None:
        excl = torch.as_tensor(exclude, dtype=torch.int64).reshape(-1).to(dev).contiguous()
        if excl.numel() != nq:
            raise ValueError("exclude: expected one row (or -1) per query (%d), got %d" % (nq, excl.numel()))
    masks = None if label_mask is None else _label_masks(label_mask, nq, dev)
    eps_t = _eps_for(stores, comm, wts, eps, q_res)
    return wts, a_op, q_raw, q_norm, nq, ms, excl, masks, eps_t


def _device_ctx(dev):
    import contextlib
    return torch.cuda.device(dev) if dev.type == "cuda" else contextlib.nullcontext()


def _range_select(exact, cand, idx_offset, excl, ms, counts=None, off=None, max_len=0, out_s=None, out_i=None,
                  after=None):
    """xmve_range_select over one shard's rescored lists.  Count mode (``off`` None) -> int64 ``[rows]`` matches per
    row.  Fill mode: the ``counts[r]`` matches of row r, sorted, to ``out_s`` / ``out_i`` ``[off[r], off[r] +
    counts[r])``; ``max_len`` >= every ``counts[r]``.  ``after`` (int64 ``[rows]``, :func:`similar_pairs_shards`):
    xmve_pair_select, which also drops every global row ``<= after[r]``."""
    cand_count, _, cand_idx = cand
    rows, cap = cand_idx.shape
    st = N.stream_ptr()
    fn, tail = ("xmve_range_select", ()) if after is None else ("xmve_pair_select", (N.ptr(after),))
    if off is None:
        counts = torch.empty((rows,), dtype=torch.int64, device=exact.device)
        if rows:
            N.call(fn, N.ptr(exact), N.ptr(cand_idx), N.ptr(cand_count), rows, cap, int(idx_offset),
                   N.ptr(excl), N.ptr(ms), N.ptr(counts), None, 0, None, None, None, *tail, st)
        return counts
    scratch = None
    if max_len > RANGE_SMEM_MAX:
        scratch = torch.empty((24 * out_s.numel(),), dtype=torch.uint8, device=exact.device)
    if rows and max_len:
        N.call(fn, N.ptr(exact), N.ptr(cand_idx), N.ptr(cand_count), rows, cap, int(idx_offset),
               N.ptr(excl), N.ptr(ms), N.ptr(counts), N.ptr(off), int(max_len), N.ptr(scratch), N.ptr(out_s),
               N.ptr(out_i), *tail, st)


def _range_merge(score, idx, seg_off, off, max_len, out_s, out_i):
    """xmve_range_merge: the sorted runs ``score`` / ``idx [seg_off[s, r], seg_off[s, r + 1])`` of every segment s
    -> row r of the CSR ``out_s`` / ``out_i`` at ``off``."""
    n_seg, rows = seg_off.shape[0], seg_off.shape[1] - 1
    if rows and max_len:
        N.call("xmve_range_merge", N.ptr(score), N.ptr(idx), n_seg, N.ptr(seg_off), rows, N.ptr(off), int(max_len),
               N.ptr(out_s), N.ptr(out_i), N.stream_ptr())


def _pow2(x):
    return 1 << max(0, int(x) - 1).bit_length()


def range_search_shards(stores, queries, min_score, weights=None, exclude=None, label_mask=None, eps=None, stats=None,
                        comm=None):
    """Range search over a corpus cut into shards (:meth:`CorpusStore.range_search` is the one-shard case; ``comm`` as
    in :func:`search_shards`, every rank passes the same queries and gets the same :class:`RangeResult`).

    1. K1 on the queries; the error bound ``eps`` (``|approx - exact| <= eps``).
    2. ``lo = round_down(min_score - 1.001 eps - 1e-7)``: a row with exact score >= min_score has an approximate score
       above ``lo``.
    3. K2 FILTER at ``lo`` over every shard, ``RANGE_CAP0`` entries per list.  The FILTER counts past the capacity, so
       the maximum over shards of every list's length is known exactly after one all-gather of the counts.
    4. rows whose list overflowed are re-run with their own capacity (the next power of two of that length), in
       passes of at most ``RANGE_PASS_ENTRIES`` list entries.  All ranks take the same decisions from the same counts.
    5. exact fp64 rescore of every listed candidate; ``xmve_range_select`` counts the rows with exact >= min_score.
    6. one shard: cumsum, fill the sorted lists, done.  Several: the counts are gathered, every rank fills its
       shards' runs into one packed block, the blocks are gathered and ``xmve_range_merge`` joins the runs.

    ``stats`` (a dict) receives eps, candidates and results per query, re-run rows and passes, and ``phases_ms``.
    The output size depends on the data, so the host reads the counts: a range search is never deferred or captured.
    There is no ``n_total`` (``search_shards`` takes one): nothing here depends on the global row count.
    """
    comm = comm or SoloComm()
    with _device_ctx(stores[0].device):
        return _range_search(stores, queries, min_score, weights, exclude, label_mask, eps, stats, comm)


def _range_search(stores, queries, min_score, weights, exclude, label_mask, eps, stats, comm, after=None, held=None):
    """``after`` and ``held``: one block of :func:`similar_pairs_shards` -- row r keeps only the global rows above
    ``after[r]``; ``held`` pairs found by the earlier blocks are counted into the memory check."""
    ref = stores[0]
    dev = ref.device
    ph = _Phases(stats is not None and dev.type == "cuda")
    ph.mark("start")
    wts, a_op, q_raw, q_norm, nq, ms, excl, masks, eps_t = _range_setup(stores, queries, min_score, weights, exclude,
                                                                        label_mask, eps, comm)
    if nq == 0:
        return RangeResult(torch.zeros((1,), dtype=torch.int64, device=dev),
                           torch.empty((0,), dtype=torch.float64, device=dev),
                           torch.empty((0,), dtype=torch.int64, device=dev))
    # 2: the FILTER floor, rounded down so that exact >= min_score implies approx > lo
    x = ms - (1.001 * eps_t.double() + 1e-7)
    lo = x.float()
    lo = torch.where(lo.double() > x, torch.nextafter(lo, torch.full_like(lo, float("-inf"))), lo)
    ph.mark("prepare_queries")
    n_st = len(stores)
    solo = n_st * comm.world == 1

    def sub(t, rows, dim=0):
        if t is None or rows is None:
            return t
        return t.index_select(dim, rows).contiguous()

    def filter_pass(rows, cap):
        """FILTER over every local store for ``rows`` (None: all) -> (per-store lists, all-shard max count, host)."""
        if rows is None:
            a_sub, n_sub = a_op, nq
        else:
            n_sub = rows.numel()
            a_sub = torch.zeros((_round_up(n_sub, _BM), ref.k), dtype=a_op.dtype, device=dev)
            a_sub[:n_sub] = a_op[rows]
        kw = {} if masks is None else {"label_mask": sub(masks, rows)}
        cands = [s._filter(a_sub, n_sub, sub(lo, rows), cap, **kw) if s.n else None for s in stores]
        cnt = torch.stack([c[0] if c is not None else torch.zeros((n_sub,), dtype=torch.int32, device=dev)
                           for c in cands])
        allc = _segments(list(cnt.unbind(0)), comm).to("cpu", torch.int64)        # one collective; host sync
        return cands, allc

    # 3: first pass
    cands, allc = filter_pass(None, RANGE_CAP0)
    need = allc.max(dim=0).values                                                   # longest list per row
    bound = int(allc.sum())                                                         # >= the number of results
    todo = torch.nonzero(need > RANGE_CAP0).flatten()
    ph.mark("filter")
    if dev.type == "cuda":
        # what the call still allocates, at most: the re-run lists (scores + rows + fp64 rescore, 16 B per entry and
        # local store, all kept until the fill) and the first pass's rescore; 16 B per result for the output and 24 B
        # for the sort scratch of the block it is filled into; sharded, the block is padded to the largest rank's
        # candidates and gathered from every rank
        n_loc = sum(1 for s in stores if s.n)
        want = 16 * n_loc * (sum(_pow2(int(c)) for c in need[todo]) + nq * RANGE_CAP0) + 16 * bound
        if solo:
            want += 24 * bound
        else:
            block = int(allc.sum(1).view(comm.world, n_st).sum(1).max())
            want += (24 + 16 + 16 * comm.world) * block
        free = torch.cuda.mem_get_info(dev)[0] + torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
        if held is not None:
            want += 16 * (held + bound) + 8 * nq                    # the final concatenation of every block's lists
            if want > free:
                raise MemoryError(
                    "similar_pairs: %d pairs found so far and up to %d more in the next %d rows need %.1f GB of device "
                    "memory for the lists, their buffers and the final result, but only %.1f GB are free on %s; raise "
                    "min_score" % (held, bound, nq, want / 1e9, free / 1e9, dev))
        if want > free:
            raise MemoryError(
                "range_search: up to %d results (%.1f per query) need %.1f GB of device memory for the lists and their "
                "buffers, but only %.1f GB are free on %s; range_count gives the exact counts without listing the "
                "rows -- raise min_score or split the queries" % (bound, bound / nq, want / 1e9, free / 1e9, dev))
    # pieces: (rows or None, per-store lists, cap); the last piece holding a row owns it.  The first pass's lists of
    # the rows that are re-run are emptied, so that they are not rescored.
    if todo.numel():
        over = torch.zeros((nq,), dtype=torch.bool)
        over[todo] = True
        over = over.to(dev)
        for c in cands:
            if c is not None:
                c[0].masked_fill_(over, 0)
    pieces = [(None, cands, RANGE_CAP0)]
    owner = torch.zeros((nq,), dtype=torch.int64)
    passes = rerun_rows = 0
    # 4: re-run the overflowed rows with lists sized from their exact counts
    while todo.numel():
        passes += 1
        if passes > RANGE_PASSES:
            raise N.XmveError("range_search: %d list(s) still overflow after %d re-run passes"
                              % (todo.numel(), RANGE_PASSES))
        rerun_rows += int(todo.numel())
        caps = torch.tensor([_pow2(int(c)) for c in need[todo]], dtype=torch.int64)
        nxt = []
        for cap in sorted(set(caps.tolist())):
            rows_c = todo[caps == cap]
            per_pass = max(1, RANGE_PASS_ENTRIES // cap)
            for r0 in range(0, rows_c.numel(), per_pass):
                rows = rows_c[r0:r0 + per_pass]
                cs, allc_r = filter_pass(rows.to(dev), cap)
                got = allc_r.max(dim=0).values
                need[rows] = got
                nxt.append(rows[got > cap])
                owner[rows] = len(pieces)
                pieces.append((rows.to(dev), cs, cap))
        todo = torch.cat(nxt)
    ph.mark("rerun")
    # 5: rescore every listed candidate, count the matches (rows a later piece owns count 0 here)
    counts = torch.zeros((n_st, nq), dtype=torch.int64, device=dev)
    done = []
    for p, (rows, cs, cap) in enumerate(pieces):
        own = (owner == p) if rows is None else (owner[rows.cpu()] == p)
        own = own.to(dev)
        q_sub, qn_sub, n_sub = sub(q_raw, rows), sub(q_norm, rows, 1), nq if rows is None else rows.numel()
        ex_sub, ms_sub = sub(excl, rows), sub(ms, rows)
        fl = {} if after is None else {"after": sub(after, rows)}
        ex_p = []
        for li, (s, c) in enumerate(zip(stores, cs)):
            if c is None:
                ex_p.append(None)
                continue
            e = s._rescore(q_sub, qn_sub, n_sub, wts, c, None)
            cp = torch.where(own, _range_select(e, c, s.index_offset, ex_sub, ms_sub, **fl),
                             torch.zeros((), dtype=torch.int64, device=dev))
            if rows is None:
                counts[li] += cp
            else:
                counts[li].index_add_(0, rows, cp)
            ex_p.append((e, cp))
        done.append((rows, cs, cap, ex_sub, ms_sub, fl, ex_p))
    ph.mark("rescore_count")

    def fill(li, s, starts, out_s, out_i):
        """Fill store ``li``'s matches of every piece; row r's run starts at ``starts[r]``."""
        for rows, cs, cap, ex_sub, ms_sub, fl, ex_p in done:
            if ex_p[li] is None:
                continue
            e, cp = ex_p[li]
            max_len = min(cap, int(counts_h[li].max())) if rows is None else min(cap, int(counts_h[li][rows.cpu()].max()))
            _range_select(e, cs[li], s.index_offset, ex_sub, ms_sub, counts=cp, off=sub(starts, rows), max_len=max_len,
                          out_s=out_s, out_i=out_i, **fl)

    # 6: lay the lists out
    if solo:
        counts_h = counts.cpu()                                                                     # host sync
        off_h = torch.zeros((nq + 1,), dtype=torch.int64)
        off_h[1:] = torch.cumsum(counts_h[0], 0)
        total = int(off_h[-1])
        off = off_h.to(dev)
        out_s = torch.empty((total,), dtype=torch.float64, device=dev)
        out_i = torch.empty((total,), dtype=torch.int64, device=dev)
        fill(0, ref, off[:-1], out_s, out_i)
    else:
        counts_h = counts.cpu()
        allc = _segments(list(counts.unbind(0)), comm).cpu()                       # [G * L, nq]: one collective
        off_h = torch.zeros((nq + 1,), dtype=torch.int64)
        off_h[1:] = torch.cumsum(allc.sum(0), 0)
        total = int(off_h[-1])
        seg_tot = allc.sum(1).view(comm.world, n_st)
        block_len = max(1, int(seg_tot.sum(1).max()))                              # padded to the largest rank's
        # this rank's block: [scores fp64 | rows int64], each block_len long; store li's runs from base[li]
        block = torch.empty((2 * block_len,), dtype=torch.int64, device=dev)
        b_s, b_i = block[:block_len].view(torch.float64), block[block_len:]
        loc_tot = counts_h.sum(1)
        base = torch.cumsum(loc_tot, 0) - loc_tot
        for li, s in enumerate(stores):
            starts = torch.cumsum(counts_h[li], 0) - counts_h[li] + base[li]
            fill(li, s, starts.to(dev), b_s, b_i)
        ph.mark("fill")
        gathered = block.unsqueeze(0) if comm.world == 1 else comm.gather(block)   # [G, 2 * block_len]
        # run (segment g * L + l, row r) starts at g * 2 block_len + (store l's base on rank g) + its offset
        seg_base = (torch.cumsum(seg_tot, 1) - seg_tot) + (torch.arange(comm.world) * 2 * block_len)[:, None]
        seg_off = torch.zeros((comm.world * n_st, nq + 1), dtype=torch.int64)
        seg_off[:, 1:] = torch.cumsum(allc, 1)
        seg_off += seg_base.reshape(-1, 1)
        flat = gathered.reshape(-1)
        off = off_h.to(dev)
        out_s = torch.empty((total,), dtype=torch.float64, device=dev)
        out_i = torch.empty((total,), dtype=torch.int64, device=dev)
        _range_merge(flat.view(torch.float64), flat[block_len:], seg_off.to(dev), off,
                     int((off_h[1:] - off_h[:-1]).max()), out_s, out_i)
    ph.mark("select_merge")
    if stats is not None:
        stats["eps"] = float(eps_t)
        stats["cap"] = RANGE_CAP0
        stats["candidates_per_query"] = bound / nq
        stats["rerun_rows"] = rerun_rows
        stats["passes"] = passes
        stats["results_per_query"] = total / nq
        stats["phases_ms"] = ph.result()
    return RangeResult(off, out_s, out_i)


def range_count_shards(stores, queries, min_score, weights=None, exclude=None, label_mask=None, eps=None, comm=None,
                       cap=8192, stats=None):
    """int64 ``[nq]`` on the device: the length of every :func:`range_search_shards` list for the same arguments,
    without listing the rows.  :func:`rank_of_gt`'s count with ``s = min_score`` and ``g = INT64_MAX``: rows whose
    approximate score is more than eps above ``min_score`` are counted by the FILTER, the rows within eps of it
    (at most ``cap`` per query; beyond, an exact fp64 pass) are rescored and compared exactly; ONE all-reduce adds
    the shards.  An excluded row is subtracted where its exact score reaches ``min_score`` (and its label is
    allowed).  No ``n_total``, as for :func:`range_search_shards`."""
    comm = comm or SoloComm()
    stores = list(stores) if isinstance(stores, (list, tuple)) else [stores]
    with _device_ctx(stores[0].device):
        wts, a_op, q_raw, q_norm, nq, ms, excl, masks, eps_t = _range_setup(stores, queries, min_score, weights,
                                                                            exclude, label_mask, eps, comm)
        dev = stores[0].device
        if nq == 0:
            return torch.zeros((0,), dtype=torch.int64, device=dev)
        live = [s for s in stores if s.n]
        g = torch.full((nq,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=dev)
        count, n_deep = _count_before_all(live, comm, a_op, q_raw, q_norm, nq, wts, ms, g, eps_t, cap, masks)
        if excl is not None:
            s_ex = comm.max_(_row_scores(live, q_raw, q_norm, nq, wts, excl, masks))
            count = count - ((s_ex > float("-inf")) & (s_ex >= ms)).to(torch.int64)
        if stats is not None:
            stats["eps"] = float(eps_t)
            stats["deep_entries"] = n_deep
        return count


#: similar pairs: the stored rows are walked in blocks of this many query rows.  8192 x 2048 bf16 rows is one FILTER
#: super-block, so each corpus line streams from HBM once per block.
PAIR_BLOCK = 8192


def similar_pairs_shards(stores, min_score, weights=None, eps=None, stats=None, comm=None):
    """Every pair of corpus rows ``i < j`` whose exact fused score reaches ``min_score`` (one float), each pair once,
    over a corpus cut into shards (:meth:`CorpusStore.similar_pairs` is the one-shard case; ``comm`` as in
    :func:`search_shards`, every rank gets the same result) -> :class:`RangeResult` with one list per global row ``i <
    N``, ``N`` the largest ``index_offset + n`` of all shards (rows no shard holds get empty lists).  Row ``i``'s list
    holds the rows ``j > i`` with ``s(i, j) >= min_score``, sorted by (score desc, j asc); ``s(i, j)`` is the score
    :func:`range_search_shards` gives row ``j`` for the stored row ``i`` as the query.

    1. the global rows are cut into blocks of ``PAIR_BLOCK`` rows, none spanning two shards; every rank derives the
       same schedule from one gather of every shard's ``(index_offset, n)``.
    2. a block's queries are its rows' stored fp32 ``raw`` rows (K1 applies the weights as for any query batch).  With
       several ranks the owner's rows reach the others through one all-reduce(sum) of a zero-filled buffer that only
       the owner fills, so the sum is exact.
    3. every shard scans only its rows ``j >= r0`` (a suffix view, :meth:`CorpusStore._suffix`); the wasted lower half
       of the diagonal block is ``PAIR_BLOCK / n`` of the work.  The range pipeline (:func:`range_search_shards`: the
       FILTER at ``round_down(min_score - 1.001 eps - 1e-7)``, the re-run from exact counts, the fp64 rescore, the
       count gather and merge) runs on those views, with ``xmve_pair_select`` keeping only ``j > i``.  eps bounds the
       residuals of every stored row, a superset of the scanned ones.
    4. the blocks' lists are appended.  Before a block allocates, the memory it needs, the pairs found so far and the
       final concatenation are checked against the free device memory: an output that cannot fit raises a sized
       ``MemoryError``.

    ``stats`` (a dict) receives eps (the largest of the blocks'), blocks, candidates, pairs, re-run rows and passes,
    and ``phases_ms`` summed over the blocks."""
    comm = comm or SoloComm()
    stores = list(stores) if isinstance(stores, (list, tuple)) else [stores]
    with _device_ctx(stores[0].device):
        return _similar_pairs(stores, min_score, weights, eps, stats, comm)


def _similar_pairs(stores, min_score, weights, eps, stats, comm):
    ms = float(min_score)
    if math.isnan(ms):
        raise ValueError("min_score: NaN")
    ref = stores[0]
    dev = ref.device
    d_all = sum(ref.dims)
    shards = _segments([torch.tensor([s.index_offset, s.n], dtype=torch.int64, device=dev) for s in stores],
                       comm).cpu()                                            # [G * L, 2]: one collective
    n_all = int((shards[:, 0] + shards[:, 1]).max())
    blocks = sorted((r0, min(o + n, r0 + PAIR_BLOCK)) for o, n in shards.tolist() for r0 in range(o, o + n, PAIR_BLOCK))
    counts = torch.zeros((n_all,), dtype=torch.int64, device=dev)
    scores, idx = [], []
    held = 0
    tot = {"eps": 0.0, "blocks": len(blocks), "candidates": 0, "pairs": 0, "rerun_rows": 0, "passes": 0,
           "phases_ms": {}}
    for r0, r1 in blocks:
        owner = [s for s in stores if s.index_offset <= r0 < s.index_offset + s.n]
        if comm.world == 1:
            q = owner[0].raw[r0 - owner[0].index_offset: r1 - owner[0].index_offset, :d_all]
        else:
            q = torch.zeros((r1 - r0, d_all), dtype=torch.float32, device=dev)
            if owner:
                q.copy_(owner[0].raw[r0 - owner[0].index_offset: r1 - owner[0].index_offset, :d_all])
            q = comm.sum_(q)
        views = [s._suffix(max(0, r0 - s.index_offset)) for s in stores]
        after = torch.arange(r0, r1, dtype=torch.int64, device=dev)
        st = None if stats is None else {}
        res = _range_search(views, q, ms, weights, None, None, eps, st, comm, after=after, held=held)
        counts[r0:r1] = res.offsets[1:] - res.offsets[:-1]
        scores.append(res.scores)
        idx.append(res.idx)
        held += res.idx.numel()
        if st is not None:
            tot["eps"] = max(tot["eps"], st["eps"])
            tot["candidates"] += int(round(st["candidates_per_query"] * (r1 - r0)))
            tot["rerun_rows"] += st["rerun_rows"]
            tot["passes"] += st["passes"]
            for k, v in st["phases_ms"].items():
                tot["phases_ms"][k] = tot["phases_ms"].get(k, 0.0) + v
    off = torch.zeros((n_all + 1,), dtype=torch.int64, device=dev)
    off[1:] = torch.cumsum(counts, 0)
    out_s = torch.cat(scores) if scores else torch.empty((0,), dtype=torch.float64, device=dev)
    out_i = torch.cat(idx) if idx else torch.empty((0,), dtype=torch.int64, device=dev)
    if stats is not None:
        tot["pairs"] = held
        stats.update(tot)
    return RangeResult(off, out_s, out_i)


def search_norm_score(stores, queries, k, weights=None, comm=None, n_total=None, **kw):
    """Top-``k`` under ``norm_score`` fusion (SURVEY.md section 8a rows A4 / F): every space's score matrix is
    min-max normalised over the WHOLE matrix (LINAS-engine/validate.py:7-11) before the weighted sum,
    ``fused[q, v] = sum_s w_s * (cos_s[q, v] - min_s) / (max_s - min_s)``.

    For corpora whose matrices cannot exist this is an affine map of the cosines, so the ranking equals that of a
    weighted-cosine search with ``w_s / (max_s - min_s)``; the global extremes are exact: ``max_s`` is the largest
    top-1 score of a one-hot search of space s, ``min_s`` minus the largest top-1 score of the negated queries.
    Costs ``2 S`` extra top-1 searches.  Returns ``(fused scores fp64 [nq, k], idx)``; the errors the reference
    would rank are ``-fused``.  ``label_mask`` is refused: the normalisation spans the whole matrix, so a filtered
    variant needs a definition of its own."""
    if kw.get("label_mask") is not None:
        raise ValueError("search_norm_score: label_mask is not supported (norm_score normalises over every row)")
    stores = list(stores) if isinstance(stores, (list, tuple)) else [stores]
    ref = stores[0]
    n_space = len(ref.dims)
    wts = _weights(weights, n_space)
    q_dev = [_to_device(x, ref.device) for x in _as_spaces(queries, ref.dims)]
    q_all = q_dev[0] if n_space == 1 else torch.cat(q_dev, dim=-1)
    adj, shift = [], 0.0
    kw_ext = {key: v for key, v in kw.items() if key not in ("exclude", "stats", "defer")}   # extremes: all rows count
    kw.pop("defer", None)
    for s in range(n_space):
        onehot = [1.0 if t == s else 0.0 for t in range(n_space)]
        top, _ = search_shards(stores, q_all, 1, weights=onehot, comm=comm, n_total=n_total, **kw_ext)
        bot, _ = search_shards(stores, -q_all, 1, weights=onehot, comm=comm, n_total=n_total, **kw_ext)
        hi, lo = float(top.max()), -float(bot.max())            # global extremes of cos_s over all (q, v)
        rng = hi - lo                                            # s / np.max(s) after s -= np.min(s)
        if not rng > 0.0:
            raise ValueError("search_norm_score: space %d has a constant score matrix (max == min); norm_score "
                             "divides by zero there, as the reference's would (validate.py:10)" % s)
        adj.append(wts[s] / rng)
        shift += wts[s] * lo / rng
    scores, idx = search_shards(stores, q_all, k, weights=adj, comm=comm, n_total=n_total, **kw)
    return scores - shift, idx


def _merge(scores, idx, k, thr=None, eps=0.0, overflow=None):
    """K3 on ``[nq, m]`` (score, global index) pairs -> top-``k`` (+ certificate when ``thr`` is given)."""
    nq, m = scores.shape
    out_s = torch.empty((nq, k), dtype=torch.float64, device=scores.device)
    out_i = torch.empty((nq, k), dtype=torch.int64, device=scores.device)
    cert = thr_next = None
    if thr is not None:
        cert = torch.empty((nq,), dtype=torch.int32, device=scores.device)
        thr_next = torch.empty((nq,), dtype=torch.float32, device=scores.device)
    if nq:
        N.call("xmve_select_topk_i64", N.ptr(scores), N.ptr(idx), nq, m, None, k, N.ptr(thr), float(eps), None,
               N.ptr(overflow), N.ptr(out_s), N.ptr(out_i), None, N.ptr(cert), N.ptr(thr_next), None, N.stream_ptr())
    if thr is None:
        return out_s, out_i
    return out_s, out_i, cert, thr_next


def _cumsum(xs):
    t = 0
    for x in xs:
        t += x
        yield t


def _weights(weights, n_space):
    if weights is None:
        return [1.0] * n_space if n_space == 1 else [1.0 / n_space] * n_space
    w = [float(x) for x in weights]
    assert len(w) == n_space, "one fusion weight per embedding space"
    return w


def merge_topk(scores, idx, k):
    """K3: ``scores/idx [G, nq, kk]`` gathered from G shards -> global top-``k`` (same ordering rule)."""
    g, nq, kk = scores.shape
    s = scores.permute(1, 0, 2).reshape(nq, g * kk).contiguous()
    i = idx.permute(1, 0, 2).reshape(nq, g * kk).contiguous()
    return _merge(s, i, k)
