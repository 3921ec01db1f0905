"""Search on corpora of at most ``SMALL_NV`` rows (B200 only): the fp64 DMMA score matrix picks candidates, the
rescore kernel scores them, and the filtered path's certified selection and re-run finish the job.

Covered: oracle parity at the selection kernel's switch points (148 / 149 / 296 / 297 / 511 / 512 query rows,
corpora of 1 000 to 16 384 rows and one past it, k from 1 to past n, one and two spaces, both norm modes, exclusions,
label masks, several stores); float-tied scores past the selection's sort; ``GraphSearch`` on small stores; agreement
with ``range_search``, ``range_count`` and ``rank_of_gt`` at ulp-level near-ties; the selection kernel without a
threshold; the bound ``small_delta`` against the measured difference of the two fp64 scores;
and memory that does not grow with the query count.  Oracle: ``oracle/linas.py`` in fp64, indices exactly, scores
within 1e-13."""
import numpy as np
import pytest
import torch

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


def _oracle_scores(V, Q, dims, w, mode="plain"):
    """fp64 scores [nq, nv]: ``-fused_errors`` (plain), or the same with ``x / max(|x|, 1e-12)`` (eps)."""
    V64, Q64 = V.astype(np.float64), Q.astype(np.float64)
    offs = np.cumsum((0,) + tuple(dims))
    if mode == "plain":
        return -linas.fused_errors([V64[:, a:b] for a, b in zip(offs[:-1], offs[1:])],
                                   [Q64[:, a:b] for a, b in zip(offs[:-1], offs[1:])], w)
    acc = None
    for (a, b), wi in zip(zip(offs[:-1], offs[1:]), w):
        qn = Q64[:, a:b] / np.maximum(np.linalg.norm(Q64[:, a:b], axis=1, keepdims=True), 1e-12)
        vn = V64[:, a:b] / np.maximum(np.linalg.norm(V64[:, a:b], axis=1, keepdims=True), 1e-12)
        e = wi * (qn @ vn.T)
        acc = e if acc is None else acc + e
    return acc


def _oracle_topk(S, k, exclude=None, allowed=None):
    """(score desc, row asc) top-k of the eligible rows, padded with -1 / -inf."""
    S = S.copy()
    if allowed is not None:
        S[~allowed] = -INF
    if exclude is not None:
        q = np.nonzero(exclude >= 0)[0]
        S[q, exclude[q]] = -INF
    idx = np.argsort(-S, axis=1, kind="stable")[:, :k]
    s = np.take_along_axis(S, idx, axis=1)
    idx = np.where(s == -INF, -1, idx)
    if idx.shape[1] < k:
        pad = k - idx.shape[1]
        idx = np.concatenate([idx, np.full((len(S), pad), -1)], axis=1)
        s = np.concatenate([s, np.full((len(S), pad), -INF)], axis=1)
    return idx, s


def _assert_oracle(s, i, ref_idx, ref_s):
    np.testing.assert_array_equal(i.cpu().numpy(), ref_idx)
    np.testing.assert_allclose(s.cpu().numpy(), ref_s, rtol=0, atol=1e-13)


def _masks(rng, nq, labels):
    """One label mask per query over labels 0..7: random subsets, every label (-1) and none (0)."""
    m = rng.integers(1, 256, nq).astype(np.int64)
    m[::7] = -1
    m[3::11] = 0
    allowed = ((m[:, None] >> labels[None, :]) & 1) == 1
    return m, allowed


def _stores(X, V, dims, mode, labels, split):
    """One store, or consecutive stores of the given sizes (the rest in the last)."""
    cuts = [0] + list(np.cumsum(split or ())) + [len(V)]
    out = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        st = X.engine.CorpusStore(b - a, dims, norm_mode=mode, index_offset=a)
        st.add(torch.from_numpy(V[a:b]), labels=None if labels is None else labels[a:b])
        out.append(st)
    return out


# ---- 1: oracle parity at the selection's switches -----------------------------------------------------------------
CASES = [  # nq, nv, k, dims, norm mode, exclude, label mask, store sizes
    (1, 1000, 10, (1536,), "plain", False, False, None),
    (148, 2048, 50, (96, 32), "plain", True, False, None),
    (149, 2049, 100, (96, 32), "eps", False, True, None),
    (296, 12000, 512, (64,), "plain", True, False, None),
    (297, 16384, 1, (64,), "eps", True, False, None),
    (511, 16384, 100, (96, 32), "plain", True, True, None),
    (512, 12000, 512, (64,), "plain", True, True, None),
    (600, 2049, 50, (64,), "eps", False, False, None),
    (2000, 16384, 100, (64, 32), "plain", True, True, None),
    (600, 16385, 100, (64, 32), "plain", True, False, None),          # large path: the same answer
    (60, 1000, 1200, (64,), "plain", True, False, None),              # k > n
    (512, 1000, 1000, (64,), "eps", True, True, None),                # k = n, with exclusions and masks
    (600, 16384, 100, (64, 32), "plain", True, True, (5000, 6000)),   # three stores
    (149, 2049, 512, (96, 32), "eps", True, True, (1000,)),
]


@pytest.mark.parametrize("nq,nv,k,dims,mode,excl,mask,split", CASES)
def test_oracle_parity(X, nq, nv, k, dims, mode, excl, mask, split):
    rng = np.random.default_rng(nq * 7919 + nv + k)
    w = (1.0,) if len(dims) == 1 else (0.7, 0.3)
    V = X.synth.clustered(nv + 3, nv, sum(dims))
    Q = X.synth.clustered(nq + 5, nq, sum(dims))
    if mode == "eps":                                        # zero rows are defined under 'eps': all scores 0
        V[nv // 2] = 0.0
        Q[nq // 2] = 0.0
    S = _oracle_scores(V, Q, dims, w, mode)
    labels = rng.integers(0, 8, nv) if mask else None
    m, allowed = _masks(rng, nq, labels) if mask else (None, None)
    ex = None
    if excl:
        ex = rng.integers(-1, nv, nq)
        ex[::2] = np.argmax(S[::2], axis=1)                   # the best row itself, for half of the queries
    stores = _stores(X, V, dims, mode, labels, split)
    kw = dict(weights=w, exclude=None if ex is None else torch.from_numpy(ex),
              label_mask=None if m is None else torch.from_numpy(m))
    s, i = X.engine.search_shards(stores, torch.from_numpy(Q), k, **kw)
    _assert_oracle(s, i, *_oracle_topk(S, k, ex, allowed))


# ---- 2: float ties past the sort ----------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["copies", "nudged"])
def tied(request):
    """16 000 x 64 corpus in which 3 000 rows are copies of one vector u, and 600 queries u + 0.1 noise: the copies
    are every query's top 3 000.  ``copies``: exact ties.  ``nudged``: one coordinate of each copy moved up by 0-31
    float steps, so the fp64 scores take 32 distinct values that agree to float precision (the construction of
    test_gpu_store_states.py, scaled under SMALL_NV).  The reference is built from the unique vectors."""
    rng = np.random.default_rng(78)
    n, d, nq = 16_000, 64, 600
    V = rng.standard_normal((n, d)).astype(np.float32)
    u = rng.standard_normal(d).astype(np.float32)
    dup = np.sort(rng.choice(n, 3_000, replace=False))
    V[dup] = u
    Q = (u + 0.1 * rng.standard_normal((nq, d))).astype(np.float32)
    if request.param == "nudged":
        c = int(np.argmax(np.abs(u)))
        V[dup, c] = u[c] + rng.integers(0, 32, len(dup)).astype(np.float32) * np.spacing(np.abs(u[c]))
    uniq, inv = np.unique(V, axis=0, return_inverse=True)
    S = -linas.cal_error(uniq.astype(np.float64), Q.astype(np.float64))[:, inv.reshape(-1)]
    if request.param == "nudged":
        for k in (100, 512):
            ref_idx, ref_s = _oracle_topk(S, k)
            kth = ref_s[:, -1:].astype(np.float32)
            assert ((S.astype(np.float32) == kth).sum(1) > 2048).mean() > 0.8        # float ties past the sort
            assert (np.searchsorted(dup, ref_idx) >= 2048).any(axis=1).all()       # beyond the first 2 048 copies
    return V, Q, S


@pytest.mark.parametrize("n_stores,k", [(1, 100), (2, 100), (5, 512)])
def test_float_ties_past_the_sort(X, tied, n_stores, k):
    """600 query rows select with a 2 048-entry sort; 3 000 float-tied scores at the k-th must come back exact, on
    one store, on two, and on five at k = 512 (the merge then holds 2 560 entries per row)."""
    V, Q, S = tied
    split = [len(V) // n_stores] * (n_stores - 1)
    stores = _stores(X, V, (V.shape[1],), "plain", None, split)
    stats = {}
    s, i = X.engine.search_shards(stores, torch.from_numpy(Q), k, stats=stats)
    _assert_oracle(s, i, *_oracle_topk(S, k))
    assert stats.get("reruns", 0) >= 1                       # the first pass cannot certify the tied rows


# ---- 3: GraphSearch on small stores -------------------------------------------------------------------------------
@pytest.mark.parametrize("nq", [60, 600])
def test_graph_search_c1_store(X, nq):
    """A C1-like 1 000 x 1 536 store: every replay equals the eager search and the oracle, a second replay with other
    queries too, and a call after ``add`` raises."""
    d, k = 1536, 10
    V = X.synth.clustered(31, 1100, d)
    store = X.engine.CorpusStore(1100, (d,)).add(torch.from_numpy(V[:1000]))
    gs = X.engine.GraphSearch(store, nq, k, with_exclude=True)
    for seed in (32, 33):
        Q = X.synth.clustered(seed, nq, d)
        S = _oracle_scores(V[:1000], Q, (d,), (1.0,))
        ex = np.argmax(S, axis=1)
        ex[1::2] = -1
        s, i = gs(torch.from_numpy(Q), exclude=torch.from_numpy(ex))
        s_e, i_e = store.search(torch.from_numpy(Q), k, exclude=torch.from_numpy(ex))
        assert torch.equal(i, i_e) and torch.equal(s, s_e)
        _assert_oracle(s, i, *_oracle_topk(S, k, ex))
    store.add(torch.from_numpy(V[1000:]))
    with pytest.raises(RuntimeError, match="corpus changed"):
        gs(torch.from_numpy(Q), exclude=torch.from_numpy(ex))


def test_graph_search_two_stores_and_label_mask(X):
    dims, w, nq, k = (96, 32), (0.6, 0.4), 200, 50
    V = X.synth.clustered(41, 9000, sum(dims))
    labels = np.random.default_rng(42).integers(0, 8, len(V))
    stores = _stores(X, V, dims, "plain", labels, (4000,))
    gs = X.engine.GraphSearch(stores, nq, k, weights=w)
    gm = X.engine.GraphSearch(stores, nq, k, weights=w, with_label_mask=True)
    for seed in (43, 44):
        Q = X.synth.clustered(seed, nq, sum(dims))
        S = _oracle_scores(V, Q, dims, w)
        s, i = gs(torch.from_numpy(Q))
        s_e, i_e = X.engine.search_shards(stores, torch.from_numpy(Q), k, weights=w)
        assert torch.equal(i, i_e) and torch.equal(s, s_e)
        _assert_oracle(s, i, *_oracle_topk(S, k))
        m, allowed = _masks(np.random.default_rng(seed), nq, labels)
        s, i = gm(torch.from_numpy(Q), label_mask=torch.from_numpy(m))
        s_e, i_e = X.engine.search_shards(stores, torch.from_numpy(Q), k, weights=w, label_mask=torch.from_numpy(m))
        assert torch.equal(i, i_e) and torch.equal(s, s_e)
        _assert_oracle(s, i, *_oracle_topk(S, k, allowed=allowed))


def test_graph_search_float_ties(X, tied):
    """The tied corpus through a graph: the first pass is replayed, the rows it cannot certify are re-run eagerly."""
    V, Q, S = tied
    store = X.engine.CorpusStore(len(V), (V.shape[1],)).add(torch.from_numpy(V))
    gs = X.engine.GraphSearch(store, len(Q), 100)
    s, i = gs(torch.from_numpy(Q))
    _assert_oracle(s, i, *_oracle_topk(S, 100))
    s, i = gs(torch.from_numpy(Q[::-1].copy()))
    _assert_oracle(s, i, *_oracle_topk(S[::-1], 100))


# ---- 4: agreement with range_search, range_count and rank_of_gt ---------------------------------------------------
def _holds_top_k(X, store, q, k, w, lm=None, excl=None):
    """range_search(q, s[:, k-1]) starts with the top-k list bit for bit, any further entry scores exactly s[:, k-1],
    and range_count equals the list lengths."""
    s, i = store.search(q, k, weights=w, label_mask=lm, exclude=excl)
    r = s[:, k - 1].contiguous()
    res = store.range_search(q, r, weights=w, label_mask=lm, exclude=excl)
    off = res.offsets.cpu()
    for row in range(q.shape[0]):
        got_i, got_s = res.idx[off[row]:off[row + 1]], res.scores[off[row]:off[row + 1]]
        assert torch.equal(got_i[:k], i[row]) and torch.equal(got_s[:k], s[row])
        assert bool((got_s[k:] == r[row]).all())
    cnt = store.range_count(q, r, weights=w, label_mask=lm, exclude=excl)
    assert torch.equal(cnt, res.offsets[1:] - res.offsets[:-1])
    return s, i


@pytest.mark.parametrize("k", [10, 100])
def test_range_search_holds_the_top_k_small(X, k):
    dims, w = (128, 64), (0.6, 0.4)
    V = X.synth.clustered(111, 12000, sum(dims))
    Q = X.synth.clustered(112, 256, sum(dims))
    assert len(V) <= X.engine.SMALL_NV
    store = X.engine.CorpusStore(len(V), dims).add(torch.from_numpy(V))
    store.set_labels(np.arange(len(V)), np.random.default_rng(113).integers(0, 4, len(V)))
    q = torch.from_numpy(Q)
    for lm, excl in ((None, None), (0b1011, torch.arange(len(Q)) * 7)):
        _holds_top_k(X, store, q, k, w, lm, excl)


def test_near_ties_agree_across_apis(X):
    """200 copies of a row that differ only in one coordinate of about 1e-4 of the row's scale, nudged by 1-8 fp32
    steps; the queries are 0 there, so the copies' exact scores differ by 1e-14 or less.  Search's j-th hit has
    exact rank j + 1, range search and range count agree with it, and the large path returns the same list with
    bit-identical scores."""
    rng = np.random.default_rng(121)
    n, d, nq, k = 8000, 64, 64, 50
    V = rng.standard_normal((n, d)).astype(np.float32)
    v = rng.standard_normal(d).astype(np.float32)
    v[-1] = np.float32(1e-4 * np.linalg.norm(v))
    rows = np.sort(rng.choice(n, 200, replace=False))
    V[rows] = v
    V[rows, -1] = v[-1] + rng.integers(1, 9, len(rows)).astype(np.float32) * np.spacing(v[-1])
    Q = (v + 0.05 * rng.standard_normal((nq, d))).astype(np.float32)
    Q[:, -1] = 0.0
    S = _oracle_scores(V, Q, (d,), (1.0,))
    top = -np.sort(-S[:, rows], axis=1)[:, :k + 1]
    assert (np.abs(np.diff(top, axis=1)) < 1e-14).all()      # the list is a run of ulp-level near-ties
    store = X.engine.CorpusStore(n, (d,)).add(torch.from_numpy(V))
    q = torch.from_numpy(Q)
    s, i = _holds_top_k(X, store, q, k, (1.0,))
    assert bool(torch.isin(i.cpu(), torch.from_numpy(rows)).all())
    ranks = X.engine.rank_of_gt([store], q, torch.arange(0, nq * k + 1, k), i.flatten())
    assert torch.equal(ranks.cpu(), torch.arange(1, k + 1, dtype=torch.int32).repeat(nq))
    s_l, i_l = store.search(q, k, small_nv=0)
    assert torch.equal(i_l, i) and torch.equal(s_l, s)
    ex = i[:, 3].contiguous()
    s_x, i_x = _holds_top_k(X, store, q, k, (1.0,), excl=ex)
    s_lx, i_lx = store.search(q, k, exclude=ex, small_nv=0)
    assert torch.equal(i_lx, i_x) and torch.equal(s_lx, s_x)


# ---- 5: the selection kernel without a threshold (candidate lists, shard lists before a merge) ------------------
def _pmax(rows, cols, k, i64):
    p = min(1 << (cols - 1).bit_length(), 16384)
    if rows >= 512:
        p = min(p, max(2048, 1 << (4 * k - 1).bit_length()))
    if p * (16 if i64 else 12) > 220 * 1024:
        p = 8192
    return p


@pytest.mark.parametrize("i64", [False, True])
@pytest.mark.parametrize("rows", [148, 149, 296, 297, 511, 512])
def test_select_without_threshold_reports_cut_ties(X, rows, i64):
    """No threshold, a ``cert`` output: cert[r] = 1 iff every entry that can belong to the top-k fit the sort.
    Row r puts a block of pmax - 1, pmax or pmax + 1 entries -- counting the k - 1 above it -- at the k-th float-
    rounded score (distinct fp64 values, some exact duplicates).  Wherever cert = 1 the list equals a stable sort;
    n_uncertified counts the other rows."""
    N = X.N
    k, cols, off = 100, 20000, 1000
    pmax = _pmax(rows, cols, k, i64)
    rng = np.random.default_rng(rows + 17 * i64)
    score = rng.uniform(-1.0, 0.4, (rows, cols))
    score[:, ::9] = -INF
    ids = np.stack([rng.permutation(10 * cols)[:cols] for _ in range(rows)]) if i64 else \
        np.tile(np.arange(cols), (rows, 1))
    want_cert = np.ones(rows, np.int32)
    for r in range(rows):
        t = pmax - (k - 1) + (r % 3) - 1                      # entries at or above the k-th float: pmax - 1 + r % 3
        pos = rng.permutation(cols)[:k - 1 + t]
        score[r, pos[:k - 1]] = rng.uniform(0.6, 0.9, k - 1)
        tied = 0.5 + rng.integers(-1000, 1000, t) * 1e-12     # all round to 0.5f
        score[r, pos[k - 1:]] = tied
        want_cert[r] = int(k - 1 + t <= pmax)
    ex = np.full(rows, -1, np.int64)
    ex[::5] = ids[::5, 7] + (0 if i64 else off)              # one excluded entry wherever it falls
    sc = torch.from_numpy(score).cuda()
    idx_t = torch.from_numpy(ids).cuda()
    ex_t = torch.from_numpy(ex).cuda()
    out_s = torch.empty((rows, k), dtype=torch.float64, device="cuda")
    out_i = torch.empty((rows, k), dtype=torch.int64, device="cuda")
    valid = torch.empty(rows, dtype=torch.int32, device="cuda")
    cert = torch.empty(rows, dtype=torch.int32, device="cuda")
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    if i64:
        N.call("xmve_select_topk_i64", N.ptr(sc), N.ptr(idx_t), rows, cols, N.ptr(ex_t), k, None, 0.0, None, None,
               N.ptr(out_s), N.ptr(out_i), N.ptr(valid), N.ptr(cert), None, N.ptr(n_bad), N.stream_ptr())
        gid = ids
    else:
        N.call("xmve_select_topk_i32", N.ptr(sc), None, rows, cols, None, off, N.ptr(ex_t), k, None, 0.0, None, None,
               N.ptr(out_s), N.ptr(out_i), N.ptr(valid), N.ptr(cert), None, N.ptr(n_bad), N.stream_ptr())
        gid = ids + off
    torch.cuda.synchronize()
    for r in range(rows):                                    # an exclusion inside the block shortens it by one
        s_r = np.where(gid[r] == ex[r], -INF, score[r])
        n_all = int((s_r > -INF).sum())
        f = s_r.astype(np.float32)
        kth = -np.sort(-f)[k - 1]
        want_cert[r] = int(n_all <= pmax or int(((s_r > -INF) & (f >= kth)).sum()) <= pmax)
        assert int(valid[r]) == n_all
    got = cert.cpu().numpy()
    np.testing.assert_array_equal(got, want_cert)
    assert int(n_bad) == int((want_cert == 0).sum()) and 0 < int(n_bad) < rows
    for r in np.nonzero(got)[0]:
        s_r = np.where(gid[r] == ex[r], -INF, score[r])
        o = np.lexsort((gid[r], -s_r))[:k]
        np.testing.assert_array_equal(out_i[r].cpu().numpy(), gid[r][o])
        np.testing.assert_array_equal(out_s[r].cpu().numpy(), s_r[o])


# ---- the bound on |DMMA - rescore| ---------------------------------------------------------------------------------
def _dmma_scores(X, store, q, wts):
    """The small path's approximate scores [nq, n]: fp64 normalisation, DMMA dot products, weighted sum."""
    N = X.N
    _, q_raw, _, _, nq = store.prepare_queries(q, wts)
    st, acc, o = N.stream_ptr(), None, 0
    for s, d in enumerate(store.dims):
        qn = torch.empty((nq, d), dtype=torch.float64, device="cuda")
        vn = torch.empty((store.n, d), dtype=torch.float64, device="cuda")
        N.call("xmve_normalize_f64", N.ptr(q_raw[:, o:o + d]), N.F32, nq, d, q_raw.stride(0), N.ptr(qn), d,
               store.norm_mode, st)
        N.call("xmve_normalize_f64", N.ptr(store.raw[:, o:o + d]), N.F32, store.n, d, store.raw.stride(0), N.ptr(vn),
               d, store.norm_mode, st)
        sc = torch.empty((nq, store.n), dtype=torch.float64, device="cuda")
        N.call("xmve_score_f64", N.ptr(qn), nq, d, N.ptr(vn), store.n, d, d, float(wts[s]), N.ptr(sc), store.n, st)
        acc = sc if acc is None else acc.add_(sc)
        o += d
    return acc


@pytest.mark.parametrize("dims,wts,mode", [((6000,), (1.0,), "plain"), ((1536, 512), (0.6, 0.4), "eps"),
                                           ((4000, 1000, 1000), (0.5, 0.3, 0.2), "plain")])
def test_small_delta_covers_dmma_minus_rescore(X, dims, wts, mode):
    """Whole matrices, the widest raw dimension the store accepts (6 000) included, with row norms near 1e+30 and
    1e-30: max |DMMA - rescore| <= small_delta."""
    nq, n = 200, 1500
    rng = np.random.default_rng(sum(dims))
    V = X.synth.clustered(sum(dims), n, sum(dims))
    Q = X.synth.clustered(sum(dims) + 1, nq, sum(dims))
    scale = np.ones(n, np.float32)
    scale[:100], scale[100:200] = 1e30, 1e-30
    V = (V * scale[:, None] / np.linalg.norm(V, axis=1, keepdims=True)).astype(np.float32)
    Q[: nq // 4] *= np.float32(1e30)
    Q[nq // 4: nq // 2] *= np.float32(1e-30)
    assert np.isfinite(V).all() and np.isfinite(Q).all() and (np.abs(V[100:200]) > 0).any()
    store = X.engine.CorpusStore(n, dims, norm_mode=mode).add(torch.from_numpy(V))
    q = torch.from_numpy(Q).cuda()
    approx = _dmma_scores(X, store, q, wts)
    _, q_raw, q_norm, _, _ = store.prepare_queries(q, wts)
    cand = (torch.full((nq,), n, dtype=torch.int32, device="cuda"), torch.zeros((nq, n), device="cuda"),
            torch.arange(n, dtype=torch.int32, device="cuda").repeat(nq, 1))
    exact = store._rescore(q_raw, q_norm, nq, wts, cand, None)
    diff = float((approx - exact).abs().max())
    delta = X.engine.small_delta(wts, dims)
    assert diff <= delta, (diff, delta)
    assert 0.0 < diff and delta < 1e-11
    S = _oracle_scores(V, Q, dims, wts, mode)
    assert float(np.abs(exact.cpu().numpy() - S).max()) < 1e-13


# ---- 6: memory ------------------------------------------------------------------------------------------------------
def test_memory_does_not_grow_with_queries(X):
    """20 000 queries against 16 000 rows in two spaces: the fp64 matrices are formed SMALL_BATCH_BYTES at a time, so
    the peak rises by at most that plus 256 MB (queries, candidate lists, rescored scores; the whole [nq, n] fp64
    matrix alone would be 2.6 GB).  The result equals the same search in batches of 500 queries."""
    dims, w, nq, k = (64, 32), (0.7, 0.3), 20_000, 10
    V = X.synth.clustered(61, 16_000, sum(dims))
    Q = torch.from_numpy(X.synth.clustered(62, nq, sum(dims))).cuda()
    store = X.engine.CorpusStore(len(V), dims).add(torch.from_numpy(V))
    store.search(Q[:500], k, weights=w)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    s, i = store.search(Q, k, weights=w)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - base
    assert rise < X.engine.SMALL_BATCH_BYTES + (256 << 20), rise / 2 ** 20
    parts = [store.search(Q[a:a + 500], k, weights=w) for a in range(0, nq, 500)]
    assert torch.equal(i, torch.cat([p[1] for p in parts])) and torch.equal(s, torch.cat([p[0] for p in parts]))
