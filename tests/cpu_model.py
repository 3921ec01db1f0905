"""A CPU *model* of one corpus shard for protocol tests (test infrastructure, never shipped).

``engine.search_shards`` orchestrates kernels through a handful of shard-local methods and three module helpers.
``ModelShard`` restates those methods in torch-CPU arithmetic (bf16-rounded operands and fp32 scores for the
filter, fp64 for the rescore) and :func:`patch_engine` swaps the module helpers, so that the control flow of the
multi-rank pipeline -- the device-side error bound, the global threshold, the two-round rescore with its gathered
pilot, the packed gather + certified merge and the re-run loop in lockstep -- runs under the ``gloo`` backend
without a GPU.  The kernels themselves are tested on the B200.
"""
import math

import torch


def _sorted_topk(score, idx, k, exclude=None, idx_offset=0):
    """(score desc, index asc) top-k of one row's valid entries -> (scores [k], ids [k], n_valid)."""
    keep = score > float("-inf")
    if exclude is not None and exclude >= 0:
        keep &= (idx + idx_offset) != exclude
    s, i = score[keep], idx[keep] + idx_offset
    order = torch.argsort(i, stable=True)
    s, i = s[order], i[order]
    order = torch.argsort(s, descending=True, stable=True)[:k]
    out_s = torch.full((k,), float("-inf"), dtype=torch.float64)
    out_i = torch.full((k,), -1, dtype=torch.int64)
    out_s[: len(order)], out_i[: len(order)] = s[order], i[order]
    return out_s, out_i, int(keep.sum())


def _certify(kth, n_valid, k, thr, eps, overflow, bound):
    enough = n_valid >= k
    complete = thr == float("-inf") or (kth - eps >= thr)
    cert = int((not overflow) and enough and complete)
    if overflow:
        nxt = bound if bound is not None else thr
    elif enough:
        nxt = float(torch.tensor(kth, dtype=torch.float32)) - 1.0001 * eps - 1e-7
    else:
        nxt = thr - max(8.0 * eps, 0.25 * abs(thr))
    return cert, nxt


class ModelShard:
    def __init__(self, rows, dims, index_offset=0):
        self.dims, self.index_offset = tuple(dims), int(index_offset)
        self.device = torch.device("cpu")
        self.raw = rows.float()
        self.n = rows.shape[0]
        self.k = sum(dims)
        parts, o = [], 0
        self.norm = []
        for d in dims:
            x = self.raw[:, o:o + d].double()
            nrm = torch.linalg.vector_norm(x, dim=1)
            self.norm.append(nrm)
            parts.append((x / nrm[:, None]).float().bfloat16().float())
            o += d
        self.op = torch.cat(parts, dim=1) if self.n else torch.zeros((0, self.k))
        self._exact_unit = None

    # -- what search_shards calls ---------------------------------------------------------------------
    def prepare_queries(self, queries, wts):
        q = torch.as_tensor(queries).float()
        parts, res, norms, o = [], [], [], 0
        for w, d in zip(wts, self.dims):
            x = q[:, o:o + d].double()
            nrm = torch.linalg.vector_norm(x, dim=1)
            y = (w * (x / nrm[:, None]).float())
            yb = y.bfloat16().float()
            parts.append(yb)
            res.append(((y - yb) ** 2).sum(1))
            norms.append(nrm)
            o += d
        return torch.cat(parts, 1), q, torch.stack(norms), torch.stack(res).float(), q.shape[0]

    def resid_max2(self):
        o, tot = 0, torch.zeros(max(self.n, 1), dtype=torch.float64)
        for d, nrm in zip(self.dims, self.norm):
            y = (self.raw[:, o:o + d].double() / nrm[:, None]).float()
            tot[: self.n] += ((y - y.bfloat16().float()) ** 2).sum(1).double()
            o += d
        return tot.max().float()

    def _exact(self, q_raw, q_norm, wts):
        acc, o = None, 0
        for s, d in enumerate(self.dims):
            qs = q_raw[:, o:o + d].double() / q_norm[s][:, None]
            vs = self.raw[:, o:o + d].double() / self.norm[s][:, None]
            e = wts[s] * (qs @ vs.T)
            acc = e if acc is None else acc + e
            o += d
        return acc

    def _eligible(self, label_mask, step=1):
        """bool [nq, rows]: which of every ``step``-th row each query's label mask allows (None: every row).  The model
        has no labels (the filtered protocol test adds them)."""
        assert label_mask is None, "ModelShard has no row labels"
        return None

    def _exact_small(self, q_raw, q_norm, nq, k, wts, excl, label_mask=None):
        sc = self._exact(q_raw, q_norm, wts)
        ok = self._eligible(label_mask)
        if ok is not None:
            sc[~ok] = float("-inf")
        ids = torch.arange(self.n)
        rows = [_sorted_topk(sc[r], ids, k, None if excl is None else int(excl[r]), self.index_offset)
                for r in range(nq)]
        return torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows])

    def _sample(self, a_op, nq, step, label_mask=None):
        sc = (a_op[:nq].float() @ self.op[::step].T).float()
        ok = self._eligible(label_mask, step)
        if ok is not None:
            sc[~ok] = float("-inf")
        return sc

    def _filter(self, a_op, nq, lo, cap, step=1, hi=None, label_mask=None):
        sc = (a_op[:nq].float() @ self.op[::step].T).float()       # re-run passes hand over a bf16 operand
        hit = sc > lo[:, None]
        ok = self._eligible(label_mask, step)
        if ok is not None:
            hit &= ok
        if hi is not None:                                          # two-sided window: count above hi, list the rest
            above = (hit & (sc > hi[:, None])).sum(1).int()
            hit &= sc <= hi[:, None]
        count = torch.zeros(nq, dtype=torch.int32)
        c_s = torch.full((nq, cap), float("nan"), dtype=torch.float32)
        c_i = torch.zeros((nq, cap), dtype=torch.int32)
        for r in range(nq):
            h = torch.nonzero(hit[r]).flatten()
            h = h[torch.randperm(len(h), generator=torch.Generator().manual_seed(r))]   # arrival order is arbitrary
            count[r] = len(h)
            m = min(len(h), cap)
            c_s[r, :m], c_i[r, :m] = sc[r, h[:m]], h[:m].int()
        return (count, c_s, c_i) if hi is None else (above, count, c_s, c_i)

    def _rescore(self, q_raw, q_norm, nq, wts, cand, bound, bound_hi=None, exact=None):
        count, c_s, c_i = cand
        cap = c_s.shape[1]
        exact_all = self._exact(q_raw[:nq], q_norm[:, :nq], wts)
        if exact is None:
            exact = torch.full((nq, cap), float("nan"), dtype=torch.float64)
        ninf = torch.tensor(float("-inf"), dtype=torch.float64)
        for r in range(nq):
            n = min(int(count[r]), cap)
            idx = c_i[r, :n].long()
            approx = c_s[r, :n]
            hi = float("inf") if bound_hi is None else float(bound_hi[r])
            lo = float("-inf") if bound is None else float(bound[r])
            mine = (approx >= lo) & (approx < hi)
            row = exact[r, :n]
            row[mine] = exact_all[r, idx[mine]]
            row[approx < lo] = ninf
        return exact

    def _pilot_top(self, exact, cand, nq, excl, m):
        count, c_s, c_i = cand
        cap = c_s.shape[1]
        out = torch.full((nq, m), float("-inf"), dtype=torch.float64)
        for r in range(nq):
            n = min(int(count[r]), cap)
            sc = exact[r, :n]
            keep = sc > float("-inf")
            if excl is not None and int(excl[r]) >= 0:
                keep &= (c_i[r, :n].long() + self.index_offset) != int(excl[r])
            top = torch.sort(sc[keep], descending=True).values[:m]
            out[r, : len(top)] = top
        return out

    def _select(self, exact, cand, nq, k, excl, thr, eps_t, bound, out_s, out_i, certify, n_bad=None):
        count, c_s, c_i = cand
        cap = c_s.shape[1]
        eps = float(eps_t)
        cert, nxt = [], []
        for r in range(nq):
            n = min(int(count[r]), cap)
            s, i, n_valid = _sorted_topk(exact[r, :n], c_i[r, :n].long(), k, None if excl is None else int(excl[r]),
                                         self.index_offset)
            out_s[r], out_i[r] = s, i
            if certify:
                c, x = _certify(float(s[k - 1]) if n_valid >= k else float("-inf"), n_valid, k, float(thr[r]), eps,
                                int(count[r]) > cap, float(bound[r]))
                cert.append(c)
                nxt.append(x)
        if certify:
            cert = torch.tensor(cert, dtype=torch.int32)
            n_bad += int((cert == 0).sum())
            return cert, torch.tensor(nxt)
        # no threshold: whether each list is exact (the model's sort has no capacity, so only an overflow spoils it)
        return (count[:nq] <= cap).to(torch.int32), None


def patch_engine(monkeypatch_setattr):
    """Swap engine._row_kth / _row_topj / _merge for torch-CPU statements of the same contracts."""
    from cross_modal_video_engine_b200 import engine

    def kth(row, j):
        return float(torch.sort(row, descending=True).values[j - 1]) if 0 < j <= len(row) else float("-inf")

    def row_kth(vals, counts, j1, sub, j2, sub_dev=None):
        if sub_dev is not None:
            sub = sub * float(sub_dev)
        out = []
        for r in range(vals.shape[0]):
            n = vals.shape[1] if counts is None else min(int(counts[r]), vals.shape[1])
            row = vals[r, :n]
            v = kth(row, j1) - sub
            if j2 > 0:
                v = max(v, kth(row, j2))
            out.append(v)
        return torch.tensor(out, dtype=torch.float32)

    def row_topj(vals, counts, j):
        out = torch.full((vals.shape[0], j), float("-inf"), dtype=torch.float32)
        for r in range(vals.shape[0]):
            n = vals.shape[1] if counts is None else min(int(counts[r]), vals.shape[1])
            top = torch.sort(vals[r, :n], descending=True).values[:j]
            out[r, : len(top)] = top
        return out

    def merge(scores, idx, k, thr=None, eps=0.0, overflow=None):
        rows = [_sorted_topk(scores[r], idx[r], k) for r in range(scores.shape[0])]
        out_s, out_i = torch.stack([r[0] for r in rows]), torch.stack([r[1] for r in rows])
        if thr is None:
            return out_s, out_i
        cert, nxt = [], []
        for r, (s, _, n_valid) in enumerate(rows):
            c, x = _certify(float(s[k - 1]) if n_valid >= k else float("-inf"), n_valid, k, float(thr[r]), eps,
                            bool(overflow[r]) if overflow is not None else False, None)
            cert.append(c)
            nxt.append(x)
        return out_s, out_i, torch.tensor(cert, dtype=torch.int32), torch.tensor(nxt)

    def eps_device(q_res, dv2, wts, n_space, k_len):
        dq2 = float(q_res.sum(0).max())
        return torch.tensor([engine.measured_eps(math.sqrt(dq2), math.sqrt(float(dv2)), wts, n_space, k_len)],
                            dtype=torch.float32)

    def pilot_bound(lists, k, eps_t):
        n_seg, nq, m = lists.shape
        out = []
        for r in range(nq):
            row = torch.sort(lists[:, r, :].reshape(-1), descending=True).values
            kth = float(row[k - 1]) if k <= len(row) else float("-inf")
            b = torch.tensor(kth - float(eps_t), dtype=torch.float64)
            f = b.float()
            if f.double() > b:                                   # round DOWN to float
                f = torch.nextafter(f, torch.tensor(float("-inf")))
            out.append(float(f) if kth > float("-inf") else float("-inf"))
        return torch.tensor(out, dtype=torch.float32)

    def merge_packed(packed, rows, length, k, thr, eps_t, n_bad):
        views = [engine.packed_views(packed[g], rows, length) for g in range(packed.shape[0])]
        scores = torch.cat([v[0] for v in views], dim=1)
        idx = torch.cat([v[1] for v in views], dim=1)
        over = torch.stack([v[2] for v in views]).max(dim=0).values
        out_s, out_i, cert, nxt = merge(scores, idx, k, thr=thr, eps=float(eps_t), overflow=over)
        n_bad += int((cert == 0).sum())
        return out_s, out_i, cert, nxt

    def count_before(exact, cand_idx, counts, idx_offset, s_gt, g, out):
        for e in range(exact.shape[0]):
            n = min(int(counts[e]), exact.shape[1])
            x, ids = exact[e, :n], cand_idx[e, :n].long() + idx_offset
            out[e] += int(((x > s_gt[e]) | ((x == s_gt[e]) & (ids < g[e]))).sum())

    monkeypatch_setattr(engine, "_count_before", count_before)
    monkeypatch_setattr(engine, "_row_kth", row_kth)
    monkeypatch_setattr(engine, "_row_topj", row_topj)
    monkeypatch_setattr(engine, "_merge", merge)
    monkeypatch_setattr(engine, "_eps_device", eps_device)
    monkeypatch_setattr(engine, "_pilot_bound", pilot_bound)
    monkeypatch_setattr(engine, "_merge_packed", merge_packed)
