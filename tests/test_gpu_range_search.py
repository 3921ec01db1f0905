"""Range search on the B200: ``xmve_range_select`` / ``xmve_range_merge`` against torch statements, and
``range_search`` / ``range_count`` against the fp64 oracle (``oracle.linas``): the listed rows exactly, scores within
1e-12, order (score desc, row asc).  Every ``min_score`` taken from the oracle lies midway between two of its scores
at least 1e-9 apart, so the boundary is unambiguous.  Also: consistency with ``search`` on a store larger than
``SMALL_NV``, the fp64 fallback of ``range_count``, the sized ``MemoryError`` and the NCCL path on two GPUs or more."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import linas

pytestmark = pytest.mark.gpu
INF = float("inf")


@pytest.fixture(scope="module")
def X():
    from cross_modal_video_engine_b200 import _native, engine, synth
    _native.require_device()

    class NS:
        pass
    ns = NS()
    ns.__dict__.update(dict(N=_native, engine=engine, synth=synth))
    return ns


def _sorted_pairs(s, i):
    """torch statement of the order: (score desc, row asc) per row of [rows, n] (invalid entries carry -inf / big)."""
    o = torch.argsort(i, dim=1, stable=True)
    s, i = torch.gather(s, 1, o), torch.gather(i, 1, o)
    o = torch.argsort(s, dim=1, descending=True, stable=True)
    return torch.gather(s, 1, o), torch.gather(i, 1, o)


def _oracle_scores(V, Q, dims=None, weights=None):
    """fp64 oracle scores [nq, nv] (the negated errors of cal_error / fused_errors)."""
    V64, Q64 = V.astype(np.float64), Q.astype(np.float64)
    if dims is None:
        return -linas.cal_error(V64, Q64)
    offs = np.cumsum((0,) + tuple(dims))
    return -linas.fused_errors([V64[:, a:b] for a, b in zip(offs[:-1], offs[1:])],
                               [Q64[:, a:b] for a, b in zip(offs[:-1], offs[1:])], weights)


def _between(row, j):
    """A minimum that exactly the best j' >= j scores of ``row`` reach, midway between neighbours >= 1e-9 apart."""
    top = np.sort(row)[::-1]
    while j < len(top) and top[j - 1] - top[j] < 1e-9:
        j += 1
    return 0.5 * (top[j - 1] + top[j]) if j < len(top) else top[-1] - 1e-3


def _check(res, S, ms, exclude=None, eligible=None):
    """res (RangeResult) against the oracle scores S: the in-range rows exactly, scores within 1e-12, sorted."""
    off = res.offsets.cpu().numpy()
    scores, idx = res.scores.cpu().numpy(), res.idx.cpu().numpy()
    assert off[0] == 0 and len(off) == len(S) + 1 and off[-1] == len(idx)
    ms = np.broadcast_to(np.asarray(ms, dtype=np.float64), (len(S),))
    for q in range(len(S)):
        want = S[q] >= ms[q]
        if eligible is not None:
            want &= eligible[q]
        if exclude is not None and exclude[q] >= 0:
            want[exclude[q]] = False
        s, i = scores[off[q]:off[q + 1]], idx[off[q]:off[q + 1]]
        np.testing.assert_array_equal(np.sort(i), np.nonzero(want)[0], err_msg="query %d" % q)
        np.testing.assert_allclose(s, S[q, i], rtol=0, atol=1e-12)
        assert np.all((s[:-1] > s[1:]) | ((s[:-1] == s[1:]) & (i[:-1] < i[1:]))), "query %d is not sorted" % q


def _store(X, V, dims, capacity=None, labels=None):
    st = X.engine.CorpusStore(capacity or len(V), dims)
    st.add(torch.from_numpy(V), labels=labels)
    return st


# ---- kernels ------------------------------------------------------------------------------------------------------
def _select(X, exact, cand_idx, counts, idx_offset, excl, ms):
    """count + cumsum + fill through the engine helper -> (offsets, scores, idx)."""
    cand = (counts, None, cand_idx)
    cnt = X.engine._range_select(exact, cand, idx_offset, excl, ms)
    off = torch.zeros(len(cnt) + 1, dtype=torch.int64, device="cuda")
    off[1:] = torch.cumsum(cnt, 0)
    total = int(off[-1])
    out_s = torch.empty(total, dtype=torch.float64, device="cuda")
    out_i = torch.empty(total, dtype=torch.int64, device="cuda")
    X.engine._range_select(exact, cand, idx_offset, excl, ms, counts=cnt, off=off[:-1],
                           max_len=min(exact.shape[1], int(cnt.max())), out_s=out_s, out_i=out_i)
    torch.cuda.synchronize()
    return cnt, off, out_s, out_i


def test_range_select_kernel(X):
    rows, cap, off0 = 700, 40960, 1000
    g = torch.Generator(device="cuda").manual_seed(3)
    exact = torch.rand((rows, cap), generator=g, device="cuda", dtype=torch.float64)
    cand_idx = torch.argsort(torch.rand((rows, cap), generator=g, device="cuda"), dim=1).to(torch.int32) * 3
    counts = torch.randint(0, 300, (rows,), generator=g, device="cuda", dtype=torch.int32)
    ms = torch.full((rows,), 0.5, dtype=torch.float64, device="cuda")
    # rows with 0, 1, 16 384, 16 385 and ~40 000 matches (the last two sort in the scratch buffer)
    counts[0], ms[0] = 500, 2.0
    counts[1], ms[1] = 500, 0.0
    exact[1, :500] = -INF
    exact[1, 17] = 0.25
    for r, m in ((2, 16384), (3, 16385), (4, 40000)):
        counts[r], ms[r] = m, -INF
    counts[5] = cap + 77                                           # an overflowed list: only cap entries are read
    exact[6, :200] = torch.round(exact[6, :200] * 8) / 8           # exact ties, ordered by row
    exact[7, :50] = float("nan")                                   # NaN never matches
    exact[8, :300] = -INF                                          # -inf entries never match, even for -inf
    ms[8] = -INF
    ms[9] = exact[9, 3]                                            # >= is inclusive
    excl = torch.full((rows,), -1, dtype=torch.int64, device="cuda")
    excl[10] = int(cand_idx[10, 4]) + off0                         # excluded rows
    excl[4] = int(cand_idx[4, 39000]) + off0
    cnt, off, out_s, out_i = _select(X, exact, cand_idx, counts, off0, excl, ms)
    n = torch.minimum(counts.long(), torch.tensor(cap, device="cuda"))
    ids = cand_idx.long() + off0
    hit = (torch.arange(cap, device="cuda")[None, :] < n[:, None]) & (exact > -INF) & (exact >= ms[:, None]) \
        & (ids != excl[:, None])
    assert torch.equal(cnt, hit.sum(1))
    assert [int(cnt[r]) for r in (0, 1, 2, 3)] == [0, 1, 16384, 16385] and int(cnt[4]) == 39999
    ws, wi = _sorted_pairs(torch.where(hit, exact, torch.full_like(exact, -INF)),
                           torch.where(hit, ids, torch.full_like(ids, 1 << 62)))
    keep = torch.arange(cap, device="cuda")[None, :] < cnt[:, None]
    assert torch.equal(out_i, wi[keep]) and torch.equal(out_s, ws[keep])


def test_range_select_needs_scratch_for_long_rows(X):
    N = X.N
    exact = torch.zeros((1, 20000), dtype=torch.float64, device="cuda")
    cand_idx = torch.arange(20000, dtype=torch.int32, device="cuda").reshape(1, -1)
    counts = torch.full((1,), 20000, dtype=torch.int32, device="cuda")
    ms = torch.zeros(1, dtype=torch.float64, device="cuda")
    cnt = torch.full((1,), 20000, dtype=torch.int64, device="cuda")
    off = torch.zeros(1, dtype=torch.int64, device="cuda")
    out_s = torch.empty(20000, dtype=torch.float64, device="cuda")
    out_i = torch.empty(20000, dtype=torch.int64, device="cuda")
    with pytest.raises(N.XmveError, match="scratch"):
        N.call("xmve_range_select", N.ptr(exact), N.ptr(cand_idx), N.ptr(counts), 1, 20000, 0, None, N.ptr(ms),
               N.ptr(cnt), N.ptr(off), 20000, None, N.ptr(out_s), N.ptr(out_i), N.stream_ptr())


@pytest.mark.parametrize("n_seg", [1, 2, 3, 4])
def test_range_merge_kernel(X, n_seg):
    rows = 600
    g = torch.Generator().manual_seed(n_seg)
    lens = torch.randint(0, 60, (n_seg, rows), generator=g)
    lens[:, 0] = 0                                                 # a row without entries
    lens[0, 1] = 5000                                              # a long run
    if n_seg > 1:
        lens[1:, 2] = 0                                            # empty runs next to a full one
    seg_off = torch.zeros((n_seg, rows + 1), dtype=torch.int64)
    pos = 7                                                        # (runs start at an arbitrary position)
    score = torch.full((int(lens.sum()) + 100,), float("nan"), dtype=torch.float64)
    idx = torch.full_like(score, -5, dtype=torch.int64)
    perm = torch.randperm(10 ** 6, generator=g)
    used = 0
    for s in range(n_seg):
        for r in range(rows):
            m = int(lens[s, r])
            seg_off[s, r] = pos
            sc = torch.round(torch.rand(m, generator=g, dtype=torch.float64) * 50) / 50     # ties across segments
            ii = perm[used:used + m]
            used += m
            ss, si = _sorted_pairs(sc[None], ii[None])
            score[pos:pos + m], idx[pos:pos + m] = ss[0], si[0]
            pos += m
        seg_off[s, rows] = pos                                     # runs of one segment lie back to back
    off = torch.zeros(rows + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(lens.sum(0), 0)
    out_s = torch.empty(int(off[-1]), dtype=torch.float64, device="cuda")
    out_i = torch.empty(int(off[-1]), dtype=torch.int64, device="cuda")
    X.engine._range_merge(score.cuda(), idx.cuda(), seg_off.cuda(), off.cuda(), int(lens.sum(0).max()), out_s, out_i)
    torch.cuda.synchronize()
    for r in range(rows):
        parts = [(score[seg_off[s, r]:seg_off[s, r] + lens[s, r]], idx[seg_off[s, r]:seg_off[s, r] + lens[s, r]])
                 for s in range(n_seg)]
        ws, wi = _sorted_pairs(torch.cat([p[0] for p in parts])[None], torch.cat([p[1] for p in parts])[None])
        assert torch.equal(out_i[off[r]:off[r + 1]].cpu(), wi[0]) and torch.equal(out_s[off[r]:off[r + 1]].cpu(), ws[0])


# ---- end to end ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spaces", ["one", "two"])
@pytest.mark.parametrize("per_query", [False, True])
def test_range_search_matches_oracle(X, spaces, per_query):
    dims, w = ((160,), None) if spaces == "one" else ((128, 64), (0.7, 0.3))
    V = X.synth.clustered(31, 30000, sum(dims))
    Q = X.synth.clustered(32, 300, sum(dims))
    store = _store(X, V, dims)
    S = _oracle_scores(V, Q, None if spaces == "one" else dims, w)
    if per_query:
        ms = np.array([_between(S[q], 1 + (q * 37) % 400) for q in range(len(Q))])
    else:
        ms = _between(S[0], 100)
    stats = {}
    res = store.range_search(torch.from_numpy(Q), ms if per_query else float(ms), weights=w, stats=stats)
    _check(res, S, ms)
    assert stats["results_per_query"] == res.idx.numel() / len(Q) and 0 < stats["eps"] < X.engine.EPS_X1
    cnt = store.range_count(torch.from_numpy(Q), ms, weights=w)
    assert torch.equal(cnt, res.offsets[1:] - res.offsets[:-1])


def test_range_search_grown_store(X):
    """Two spaces, capacity 60 000: 25 000 rows in two ragged adds, then 15 000 more (norm planes read by stride)."""
    dims, w = (128, 64), (0.6, 0.4)
    V = X.synth.clustered(41, 40000, sum(dims))
    Q = X.synth.clustered(42, 200, sum(dims))
    store = X.engine.CorpusStore(60000, dims)
    store.add(torch.from_numpy(V[:11111]))
    store.add(torch.from_numpy(V[11111:25000]))
    for n in (25000, 40000):
        S = _oracle_scores(V[:n], Q, dims, w)
        ms = np.array([_between(S[q], 50 + q) for q in range(len(Q))])
        _check(store.range_search(torch.from_numpy(Q), ms, weights=w), S, ms)
        if n == 25000:
            store.add(torch.from_numpy(V[25000:]))


def test_range_search_edges(X):
    dims = (96,)
    V = X.synth.clustered(51, 20000, 96)
    Q = X.synth.clustered(52, 600, 96)                             # more than one 128-query tile and > 512 rows
    store = _store(X, V, dims)
    S = _oracle_scores(V, Q)
    # above every score: empty lists
    res = store.range_search(torch.from_numpy(Q), float(S.max()) + 1e-6)
    assert res.idx.numel() == 0 and torch.equal(res.offsets, torch.zeros(601, dtype=torch.int64, device="cuda"))
    ps, pi = res.padded()
    assert ps.shape == (600, 0) and pi.shape == (600, 0)
    # +inf per query, mixed with finite minima; at most 128 queries
    ms = np.array([_between(S[q], 20) for q in range(100)])
    ms[::7] = INF
    _check(store.range_search(torch.from_numpy(Q[:100]), ms), S[:100], ms)
    # exclude (rows inside the range, and -1)
    ms = np.array([_between(S[q], 30) for q in range(600)])
    excl = np.array([int(np.argsort(-S[q])[q % 30]) if q % 3 else -1 for q in range(600)])
    res = store.range_search(torch.from_numpy(Q), ms, exclude=torch.from_numpy(excl))
    _check(res, S, ms, exclude=excl)
    assert torch.equal(store.range_count(torch.from_numpy(Q), ms, exclude=torch.from_numpy(excl)),
                       res.offsets[1:] - res.offsets[:-1])
    # padded(): what search returns, -inf / -1 padded
    ps, pi = res.padded()
    lens = (res.offsets[1:] - res.offsets[:-1]).cpu()
    assert pi.shape == (600, int(lens.max()))
    for q in (0, 1, 599):
        assert torch.equal(pi[q, :lens[q]], res.idx[res.offsets[q]:res.offsets[q + 1]])
        assert bool((pi[q, lens[q]:] == -1).all()) and bool((ps[q, lens[q]:] == -INF).all())


def test_range_search_all_rows_of_a_small_store(X):
    V = X.synth.clustered(61, 3000, 64)
    Q = X.synth.clustered(62, 40, 64)
    store = _store(X, V, (64,))
    S = _oracle_scores(V, Q)
    res = store.range_search(torch.from_numpy(Q), -INF)
    _check(res, S, -INF)
    assert res.idx.numel() == 40 * 3000
    assert torch.equal(store.range_count(torch.from_numpy(Q), -INF), torch.full((40,), 3000, device="cuda"))


def test_range_search_label_mask(X):
    dims = (128,)
    V = X.synth.clustered(71, 25000, 128)
    Q = X.synth.clustered(72, 300, 128)
    labels = np.random.default_rng(73).integers(0, 64, len(V))
    store = _store(X, V, dims, labels=labels)
    S = _oracle_scores(V, Q)
    masks = np.random.default_rng(74).integers(-(1 << 62), 1 << 62, len(Q))
    masks[0], masks[1], masks[2] = -1, 0, 1 << 9                   # every label, none, one
    m = masks.view(np.uint64)
    elig = ((m[:, None] >> labels.astype(np.uint64)[None, :]) & np.uint64(1)) != 0
    ms = np.array([_between(np.where(elig[q], S[q], -1.0), 1 + q % 60) for q in range(len(Q))])
    ms[1] = -INF                                                   # mask 0: nothing, whatever the minimum
    excl = np.array([int(np.argmax(np.where(elig[q], S[q], -9))) if q % 2 else -1 for q in range(len(Q))])
    lm = torch.from_numpy(masks)
    res = store.range_search(torch.from_numpy(Q), ms, label_mask=lm, exclude=torch.from_numpy(excl))
    _check(res, S, ms, exclude=excl, eligible=elig)
    assert int(res.offsets[2] - res.offsets[1]) == 0
    for ex in (None, torch.from_numpy(excl)):
        cnt = store.range_count(torch.from_numpy(Q), ms, label_mask=lm, exclude=ex)
        want = [int((elig[q] & (S[q] >= ms[q])).sum()) - (1 if ex is not None and excl[q] >= 0 and elig[q, excl[q]]
                                                         and S[q, excl[q]] >= ms[q] else 0) for q in range(len(Q))]
        assert cnt.tolist() == want


def test_range_search_exact_duplicates(X):
    """Every corpus row three times: tied scores come back ordered by row."""
    base = X.synth.clustered(81, 7000, 64)
    V = np.concatenate([base, base, base])
    Q = X.synth.clustered(82, 150, 64)
    store = _store(X, V, (64,))
    S = _oracle_scores(V, Q)
    ms = np.array([_between(S[q], 3 * (1 + q % 20)) for q in range(len(Q))])
    res = store.range_search(torch.from_numpy(Q), ms)
    _check(res, S, ms)
    s = res.scores[res.offsets[0]:res.offsets[1]].cpu().numpy()
    assert len(s) % 3 == 0 and np.array_equal(s[0::3], s[1::3]) and np.array_equal(s[0::3], s[2::3])


def test_range_search_long_lists(X):
    """Queries with more than 2 048 results (the lists are re-run, sized from their counts) and with more than
    16 384 (sorted in the scratch buffer)."""
    V = X.synth.clustered(91, 60000, 64, n_centroid=4)
    Q = X.synth.clustered(92, 130, 64, n_centroid=4)
    store = _store(X, V, (64,))
    S = _oracle_scores(V, Q)
    depth = [20, 3000, 20000, 40000] * 33
    ms = np.array([_between(S[q], depth[q]) for q in range(len(Q))])
    stats = {}
    res = store.range_search(torch.from_numpy(Q), ms, stats=stats)
    _check(res, S, ms)
    lens = (res.offsets[1:] - res.offsets[:-1]).cpu()
    assert int(lens[1]) >= 3000 and int(lens[2]) > 16384 and stats["rerun_rows"] >= 97 and stats["passes"] == 1
    assert torch.equal(store.range_count(torch.from_numpy(Q), ms), lens.cuda())


def test_two_stores_equal_one(X):
    dims, w = (128, 64), (0.5, 0.5)
    V = X.synth.clustered(101, 36000, sum(dims))
    Q = X.synth.clustered(102, 200, sum(dims))
    one = _store(X, V, dims)
    a = X.engine.CorpusStore(20000, dims, index_offset=0).add(torch.from_numpy(V[:20000]))
    b = X.engine.CorpusStore(16000, dims, index_offset=20000).add(torch.from_numpy(V[20000:]))
    S = _oracle_scores(V, Q, dims, w)
    ms = np.array([_between(S[q], [5, 300, 3000][q % 3]) for q in range(len(Q))])
    excl = np.array([int(np.argsort(-S[q])[1]) for q in range(len(Q))])
    r1 = one.range_search(torch.from_numpy(Q), ms, weights=w, exclude=torch.from_numpy(excl))
    r2 = X.engine.range_search_shards([a, b], torch.from_numpy(Q), ms, weights=w, exclude=torch.from_numpy(excl))
    _check(r1, S, ms, exclude=excl)
    assert torch.equal(r1.offsets, r2.offsets) and torch.equal(r1.idx, r2.idx) and torch.equal(r1.scores, r2.scores)
    c2 = X.engine.range_count_shards([a, b], torch.from_numpy(Q), ms, weights=w, exclude=torch.from_numpy(excl))
    assert torch.equal(c2, r1.offsets[1:] - r1.offsets[:-1])


# ---- consistency with search --------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 1000])
def test_range_search_holds_the_top_k(X, k):
    """r[q] = the k-th score search returns: range_search(q, r) starts with exactly the top-k list; any further entry
    scores exactly r[q].  (test_gpu_small_path.py checks the same at most SMALL_NV rows.)"""
    dims, w = (128, 64), (0.6, 0.4)
    V = X.synth.clustered(111, 50000, sum(dims))
    Q = X.synth.clustered(112, 256, sum(dims))
    assert len(V) > X.engine.SMALL_NV
    store = _store(X, V, dims)
    labels = np.random.default_rng(113).integers(0, 4, len(V))
    store.set_labels(np.arange(len(V)), labels)
    q = torch.from_numpy(Q)
    for lm, excl in ((None, None), (0b1011, torch.arange(len(Q)) * 7)):
        s, i = store.search(q, k, weights=w, label_mask=lm, exclude=excl)
        r = s[:, k - 1].contiguous()
        res = store.range_search(q, r, weights=w, label_mask=lm, exclude=excl)
        off = res.offsets.cpu()
        for row in range(len(Q)):
            got_i, got_s = res.idx[off[row]:off[row + 1]], res.scores[off[row]:off[row + 1]]
            assert torch.equal(got_i[:k], i[row]) and torch.equal(got_s[:k], s[row])
            assert bool((got_s[k:] == r[row]).all())
        cnt = store.range_count(q, r, weights=w, label_mask=lm, exclude=excl)
        assert torch.equal(cnt, res.offsets[1:] - res.offsets[:-1])


def test_range_count_deep_fallback(X):
    """A band capacity of 16 rows sends most queries to the exact fp64 pass: the counts do not change."""
    dims, w = (128, 64), (0.6, 0.4)
    V = X.synth.clustered(121, 30000, sum(dims))
    Q = X.synth.clustered(122, 64, sum(dims))
    store = _store(X, V, dims)
    S = _oracle_scores(V, Q, dims, w)
    ms = np.array([_between(S[q], 500 + 40 * q) for q in range(len(Q))])
    labels = np.random.default_rng(123).integers(0, 3, len(V))
    store.set_labels(np.arange(len(V)), labels)
    q = torch.from_numpy(Q)
    for lm in (None, 0b101):
        ref = store.range_count(q, ms, weights=w, label_mask=lm)
        stats = {}
        deep = X.engine.range_count_shards([store], q, ms, weights=w, label_mask=lm, cap=16, stats=stats)
        assert stats["deep_entries"] > 0 and torch.equal(deep, ref)
        elig = np.ones(len(V), bool) if lm is None else ((lm >> labels) & 1) == 1
        assert ref.tolist() == [int(((S[j] >= ms[j]) & elig).sum()) for j in range(len(Q))]


def test_range_count_deep_fallback_with_many_ties(X):
    """Every row 100 times and min_score equal to a tied score: the fp64 fallback's band of rows within 1e-13 of the
    minimum holds 100 rows, more than its first list, and the count still equals the list length."""
    base = X.synth.clustered(141, 400, 64)
    store = _store(X, np.tile(base, (100, 1)), (64,))
    q = torch.from_numpy(X.synth.clustered(142, 16, 64))
    s, _ = store.search(q, 350)
    r = s[:, 349].contiguous()                                     # the 350th score: a 100-fold tie
    res = store.range_search(q, r)
    lens = res.offsets[1:] - res.offsets[:-1]
    assert bool((lens % 100 == 0).all()) and bool((lens >= 400).all())
    stats = {}
    deep = X.engine.range_count_shards([store], q, r, cap=16, stats=stats)
    assert stats["deep_entries"] == 16 and torch.equal(deep, lens)


def test_range_search_refuses_an_output_that_cannot_fit(X):
    """min_score = -inf for 60 000 queries over 100 000 rows: 6e9 results, 240 GB.  The call raises a sized
    MemoryError before it allocates the output."""
    V = X.synth.clustered(131, 100000, 64)
    store = _store(X, V, (64,))
    Q = torch.from_numpy(np.tile(X.synth.clustered(132, 1000, 64), (60, 1)))
    torch.cuda.reset_peak_memory_stats()
    with pytest.raises(MemoryError, match="range_count"):
        store.range_search(Q, -INF)
    assert torch.cuda.max_memory_allocated() < 40e9


def test_cli_min_score(X, tmp_path, capsys):
    """cli.py search --min-score: id lists per query (one minimum per query from a .npy), and a run file (one for all)."""
    from cross_modal_video_engine_b200 import cli, corpus_io
    V, Q, vid, _, _ = X.synth.msrvtt_like(93, 300, 2, 64, 2.0)
    corpus_io.write_bigfile(str(tmp_path / "bf"), vid, V)
    np.save(str(tmp_path / "q.npy"), Q)
    S = _oracle_scores(V, Q)
    ms = np.array([_between(S[q], 1 + q % 5) for q in range(len(Q))])
    np.save(str(tmp_path / "ms.npy"), ms)
    args = ["search", "--corpus", str(tmp_path / "bf"), "--queries", str(tmp_path / "q.npy")]
    assert cli.main(args + ["--min-score", str(tmp_path / "ms.npy")]) == 0
    lines = capsys.readouterr().out.strip().splitlines()
    assert len(lines) == len(Q)
    for q in (0, 3, len(Q) - 1):
        hit = np.nonzero(S[q] >= ms[q])[0]
        order = hit[np.lexsort((hit, -S[q, hit]))]
        assert lines[q] == str([vid[i] for i in order])
    run = tmp_path / "run.txt"
    assert cli.main(args + ["--min-score", repr(float(ms[0])), "--run-file", str(run)]) == 0
    first = [ln.split() for ln in run.read_text().splitlines() if ln.startswith("q0 ")]
    assert len(first) == int((S[0] >= ms[0]).sum()) and first[0][2] == vid[int(np.argmax(S[0]))]


# ---- several GPUs (NCCL) ------------------------------------------------------------------------------------------
def test_sharded_range_search_nccl():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two GPUs or more")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc_per_node", str(min(4, n)),
                          "--master_port", str(port), os.path.join(ROOT, "tools", "check_range_sharded.py")],
                         cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "range sharded ok" in out.stdout
