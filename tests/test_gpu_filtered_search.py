"""Filtered search (``label_mask``) on the B200: the labelled FILTER kernel and the score-mask kernel against their
unlabelled counterparts plus host-side masking, and the filtered search against the fp64 oracle restricted to the
eligible rows (``err[q, ineligible] = +inf``, output truncated to ``min(k, #eligible)``): indices exactly, scores
within 1e-13.  Also: store states (small path, partially filled then grown, ``set_labels`` between searches and right
before a head-stream search, two shards in one process), ``GraphSearch(with_label_mask=True)``, and an unfiltered
search of a labelled store equal to that of an unlabelled one.  The NCCL check runs on two GPUs or more."""
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


@pytest.fixture(scope="module")
def X():
    from cross_modal_video_engine_b200 import _native, engine, synth
    _native.require_device()

    class NS:
        pass
    ns = NS()
    ns.__dict__.update(dict(N=_native, engine=engine, synth=synth))
    return ns


def _rup(x, m):
    return (x + m - 1) // m * m


def _bits(labels):
    m = 0
    for b in labels:
        m |= 1 << int(b)
    return m - (1 << 64) if m >= (1 << 63) else m


def _allowed(masks, labels):
    """numpy [nq, nv] bool: bit labels[v] of masks[q] (int64 bit patterns) is set."""
    m = np.asarray(masks, dtype=np.int64).view(np.uint64)
    return ((m[:, None] >> labels.astype(np.uint64)[None, :]) & np.uint64(1)) != 0


def _oracle_masked(V, Q, k, labels, masks, weights=None, dims=None, exclude=None):
    """fp64 oracle over the eligible rows -> (idx int64 [nq, k] -1 padded, scores [nq, k] -inf padded)."""
    V64, Q64 = V.astype(np.float64), Q.astype(np.float64)
    if dims is None:
        err = linas.cal_error(V64, Q64)
    else:
        offs = np.cumsum((0,) + tuple(dims))
        err = linas.fused_errors([V64[:, a:b] for a, b in zip(offs[:-1], offs[1:])],
                                 [Q64[:, a:b] for a, b in zip(offs[:-1], offs[1:])], weights)
    masks = np.broadcast_to(np.asarray(masks, dtype=np.int64), (len(Q),))
    err = np.where(_allowed(masks, labels), err, np.inf)
    if exclude is not None:
        for q, e in enumerate(exclude):
            if e >= 0:
                err[q, e] = np.inf
    idx = np.argsort(err, axis=1, kind="stable")[:, :k]
    e = np.take_along_axis(err, idx, axis=1)
    valid = np.isfinite(e)
    return np.where(valid, idx, -1), np.where(valid, -e, -np.inf)


def _assert_oracle(s, i, ref_idx, ref_s):
    np.testing.assert_array_equal(i.cpu().numpy(), ref_idx)
    np.testing.assert_allclose(s.cpu().numpy(), ref_s, rtol=0, atol=1e-13)


# ---- kernels ------------------------------------------------------------------------------------------------------
def _operands(N, nq, nv, d, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn((nq, d), generator=g, device="cuda")
    v = torch.randn((nv, d), generator=g, device="cuda")
    a = torch.zeros((_rup(nq, 128), d), dtype=torch.bfloat16, device="cuda")
    b = torch.zeros((_rup(nv, 256), d), dtype=torch.bfloat16, device="cuda")
    st = N.stream_ptr()
    for x, op, n in ((q, a, nq), (v, b, nv)):
        N.call("xmve_prepare_rows", N.ptr(x), N.F32, n, d, 1, d, None, 0, 0, None, None, N.ptr(op), op.stride(0), 0,
               0, 1.0, 0, st)
    return a, b


def _filter(N, name, a, nq, b, rows, step, d, lo, hi, cap, extra=()):
    above = torch.zeros(nq, dtype=torch.int32, device="cuda")
    count = torch.zeros(nq, dtype=torch.int32, device="cuda")
    c_s = torch.zeros((nq, cap), dtype=torch.float32, device="cuda")
    c_i = torch.full((nq, cap), -1, dtype=torch.int32, device="cuda")
    N.call(name, N.ptr(a), nq, a.stride(0), N.ptr(b), rows, b.stride(0), step, d, N.ptr(lo), N.ptr(hi),
           N.ptr(above) if hi is not None else None, N.ptr(count), N.ptr(c_s), N.ptr(c_i), cap, *extra, N.stream_ptr())
    torch.cuda.synchronize()
    return above, count, c_s, c_i


@pytest.mark.parametrize("tile", ["0", "1", "4", "5"])
@pytest.mark.parametrize("single_hit", ["0", "1"])
@pytest.mark.parametrize("step", [1, 3])
def test_labeled_filter_equals_filter_then_mask(X, monkeypatch, tile, single_hit, step):
    """Same operands, same window: the labelled kernel lists exactly the eligible entries of the unlabelled list
    (as a set of (score, index) pairs, same count) and counts above hi only eligible columns."""
    N = X.N
    monkeypatch.setenv("XMVE_TILE", tile)
    monkeypatch.setenv("XMVE_SINGLE_HIT", single_hit)
    nq, nv, d = 300, 15001, 128                                   # nq % 128 != 0; sampled rows % 256 != 0
    a, b = _operands(N, nq, nv, d, seed=7)
    rows = (nv + step - 1) // step
    g = torch.Generator(device="cuda").manual_seed(8)
    labels = torch.randint(0, 64, (nv,), generator=g, device="cuda", dtype=torch.int32).to(torch.uint8)
    allow = torch.randint(-(1 << 62), 1 << 62, (nq,), generator=g, device="cuda", dtype=torch.int64)
    allow[0], allow[1], allow[2] = -1, 0, 1 << 5                  # every label, none, one
    allow[3] = allow[3] | (-(1 << 63))                            # bit 63 (label 63) set
    sc = torch.randn((nq,), generator=g, device="cuda")
    lo = (0.2 + 0.02 * sc).float()                               # unit rows, d = 128: ~1-4 % of the scores
    hi = lo + 0.05
    cap = 4096
    lab_col = labels[::step][:rows].long()
    ok = ((allow[:, None] >> lab_col[None, :]) & 1) != 0          # [nq, rows]
    for with_hi in (False, True):
        h = hi if with_hi else None
        above, count, c_s, c_i = _filter(N, "xmve_score_filter", a, nq, b, rows, step, d, lo, h, cap)
        l_above, l_count, l_s, l_i = _filter(N, "xmve_score_filter_labeled", a, nq, b, rows, step, d, lo, h, cap,
                                             (N.ptr(labels), N.ptr(allow)))
        assert int(count.max()) < cap
        if with_hi:                                               # with every label allowed: the unlabelled count
            full = torch.full_like(allow, -1)
            f_above = _filter(N, "xmve_score_filter_labeled", a, nq, b, rows, step, d, lo, h, cap,
                              (N.ptr(labels), N.ptr(full)))[0]
            assert torch.equal(f_above, above)
        for r in range(nq):
            n = int(count[r])
            idx = c_i[r, :n].long()
            keep = ok[r, idx]
            want = set(zip(c_s[r, :n][keep].tolist(), idx[keep].tolist()))
            ln = int(l_count[r])
            got = set(zip(l_s[r, :ln].tolist(), l_i[r, :ln].long().tolist()))
            assert ln == len(want) and got == want, "row %d" % r
        assert int(l_count[1]) == 0 and int(l_above[1]) == 0
        assert torch.equal(l_count[0], count[0])
    # count_above counts eligible columns only: the labelled list of the window (hi, +inf) holds exactly those
    _, c2, _, _ = _filter(N, "xmve_score_filter_labeled", a, nq, b, rows, step, d, hi, None, cap,
                          (N.ptr(labels), N.ptr(allow)))
    assert torch.equal(l_above, c2)


def test_labeled_filter_refuses_wide_tile(X, monkeypatch):
    N = X.N
    a, b = _operands(N, 128, 1000, 64, seed=3)
    lo = torch.zeros(128, device="cuda")
    labels = torch.zeros(1000, dtype=torch.uint8, device="cuda")
    allow = torch.full((128,), -1, dtype=torch.int64, device="cuda")
    for tile in ("2", "6"):
        monkeypatch.setenv("XMVE_TILE", tile)
        with pytest.raises(N.XmveError, match="wide tile"):
            _filter(N, "xmve_score_filter_labeled", a, 128, b, 1000, 1, 64, lo, None, 64,
                    (N.ptr(labels), N.ptr(allow)))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("step", [1, 4])
def test_mask_scores_matches_torch(X, dtype, step):
    N = X.N
    rows, cols, ld = 70, 3001, 3008
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn((rows, ld), generator=g, device="cuda").to(dtype)
    labels = torch.randint(0, 64, (cols * step,), generator=g, device="cuda", dtype=torch.int32).to(torch.uint8)
    allow = torch.randint(-(1 << 62), 1 << 62, (rows,), generator=g, device="cuda", dtype=torch.int64)
    allow[0] = -(1 << 63)
    want = x.clone()
    ok = ((allow[:, None] >> labels[::step][:cols].long()[None, :]) & 1) != 0
    want[:, :cols][~ok] = float("-inf")
    N.call("xmve_mask_scores", N.ptr(x), N.F32 if dtype == torch.float32 else N.F64, rows, cols, ld, N.ptr(labels),
           step, N.ptr(allow), N.stream_ptr())
    assert torch.equal(x, want)


# ---- search -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def one_space(X):
    nv, d = 200_000, 256
    V, Q = X.synth.gaussian(300, nv, d), X.synth.gaussian(301, 600, d)
    rng = np.random.default_rng(302)
    labels = rng.integers(0, 61, nv).astype(np.uint8)          # labels 0-60: ~1.6 % of the rows each
    rare = rng.choice(nv, 1030, replace=False)
    labels[rare[:1000]] = 61                                    # 0.5 % of the rows
    labels[rare[1000:]] = 62                                    # 30 rows: fewer than k
    store = X.engine.CorpusStore(nv, (d,))
    store.add(torch.from_numpy(V[:120_000]), labels=labels[:120_000]).add(torch.from_numpy(V[120_000:]),
                                                                      labels=torch.from_numpy(labels[120_000:]))
    return V, Q, labels, store


def _masks(nq, rng):
    """A different mask per query: all labels, ~30 %, ~5 %, 30 rows, 0, ~1.6 % and random 16-label masks."""
    base = [-1, _bits(range(19)), _bits(range(3)), _bits([62]), 0, _bits([62, 5])]
    out = [base[i % len(base)] if i < 60 else _bits(rng.choice(64, 16, replace=False)) for i in range(nq)]
    return np.array(out, dtype=np.int64)


@pytest.mark.parametrize("k", [100, 1000])
def test_filtered_search_one_space(X, one_space, k):
    V, Q, labels, store = one_space
    q = torch.from_numpy(Q[:300])
    s0, i0 = store.search(q, k)
    s1, i1 = store.search(q, k, label_mask=-1)                    # every label: bit for bit the unfiltered search
    assert torch.equal(i0, i1) and torch.equal(s0, s1)
    rng = np.random.default_rng(k)
    for frac_labels in (_bits(range(19)), _bits(range(3)), _bits([61])):
        s, i = store.search(q, k, label_mask=frac_labels)        # ~30 %, ~5 %, 0.5 % (one mask for the batch)
        _assert_oracle(s, i, *_oracle_masked(V, Q[:300], k, labels, frac_labels))
    masks = _masks(300, rng)
    excl = np.full(300, -1)
    excl[::7] = np.asarray(i0[::7, 0].cpu())                      # drop the unfiltered best row of some queries
    stats = {}
    s, i = store.search(q, k, label_mask=masks, exclude=torch.from_numpy(excl), stats=stats)
    _assert_oracle(s, i, *_oracle_masked(V, Q[:300], k, labels, masks, exclude=excl))
    assert stats["thr_inf_rows"] > 0 and stats["eligible_min"] == 0
    assert bool((i[4] == -1).all())                               # mask 0: all padding


def test_filtered_search_600_queries_uint64(X, one_space):
    """600 queries (the >= 512-row selection), masks given as a numpy uint64 array."""
    V, Q, labels, store = one_space
    masks = _masks(600, np.random.default_rng(9))
    s, i = store.search(torch.from_numpy(Q), 100, label_mask=masks.view(np.uint64))
    _assert_oracle(s, i, *_oracle_masked(V, Q, 100, labels, masks))


DIMS, W = (96, 32), (0.7, 0.3)


def test_filtered_search_two_spaces_and_store_states(X):
    """Two spaces with weights: a store partially filled, searched, then grown; set_labels between two searches; a
    head-stream search straight after set_labels; the <= 16 k-row path; two shards in one process."""
    V, Q, _, _, _ = X.synth.msrvtt_like(23, 60_000, 1, sum(DIMS), 2.5)
    Q = Q[:300]
    rng = np.random.default_rng(24)
    labels = rng.integers(0, 64, len(V)).astype(np.uint8)
    masks = _masks(300, rng)
    q = torch.from_numpy(Q)
    k = 100
    store = X.engine.CorpusStore(90_000, DIMS)
    store.add(torch.from_numpy(V[:25_000]), labels=labels[:25_000])
    s, i = store.search(q, k, weights=W, label_mask=masks)
    _assert_oracle(s, i, *_oracle_masked(V[:25_000], Q, k, labels[:25_000], masks, W, DIMS))
    store.add(torch.from_numpy(V[25_000:]), labels=labels[25_000:])
    s, i = store.search(q, k, weights=W, label_mask=masks)
    _assert_oracle(s, i, *_oracle_masked(V, Q, k, labels, masks, W, DIMS))
    # relabel: every row with label 7 becomes 62, and 500 random rows become 7
    new = labels.copy()
    moved = np.nonzero(labels == 7)[0]
    new[moved] = 62
    pick = rng.choice(len(V), 500, replace=False)
    new[pick] = 7
    ids = np.concatenate([moved, pick])
    ids = np.unique(ids)
    store.set_labels(ids, new[ids])
    m2 = np.array([_bits([7]), _bits([62]), _bits([7, 62])] * 100, dtype=np.int64)
    s, i = store.search(q, k, weights=W, label_mask=m2)
    _assert_oracle(s, i, *_oracle_masked(V, Q, k, new, m2, W, DIMS))
    store.set_labels(ids, labels[ids])
    head = torch.cuda.Stream()
    p = X.engine.search_shards([store], q, k, weights=W, label_mask=m2, defer=True, head_stream=head)
    s, i = p.result()
    _assert_oracle(s, i, *_oracle_masked(V, Q, k, labels, m2, W, DIMS))
    # two shards in one process equal one store
    a = X.engine.CorpusStore(30_000, DIMS).add(torch.from_numpy(V[:30_000]), labels=labels[:30_000])
    b = X.engine.CorpusStore(30_000, DIMS, index_offset=30_000).add(torch.from_numpy(V[30_000:]),
                                                                    labels=labels[30_000:])
    s2, i2 = X.engine.search_shards([a, b], q, k, weights=W, label_mask=masks)
    s1, i1 = store.search(q, k, weights=W, label_mask=masks)
    assert torch.equal(i1, i2)
    _assert_oracle(s2, i2, *_oracle_masked(V, Q, k, labels, masks, W, DIMS))
    # relabel rows of shard `a` only: set_labels is given the same global ids on every shard, each applies its own
    ids = rng.choice(30_000, 2_000, replace=False)
    relab = labels.copy()
    relab[ids] = 62
    for st_ in (a, b, store):
        st_.set_labels(ids, relab[ids])
    assert b.label_version == a.label_version and int(b.label_hist[62]) == int((labels[30_000:] == 62).sum())
    s2, i2 = X.engine.search_shards([a, b], q, k, weights=W, label_mask=masks)
    s1, i1 = store.search(q, k, weights=W, label_mask=masks)
    assert torch.equal(i1, i2) and torch.equal(s1, s2)
    _assert_oracle(s2, i2, *_oracle_masked(V, Q, k, relab, masks, W, DIMS))
    # the <= 16 k-row path
    small = X.engine.CorpusStore(12_000, DIMS).add(torch.from_numpy(V[:12_000]), labels=labels[:12_000])
    s, i = small.search(q, 50, weights=W, label_mask=masks)
    _assert_oracle(s, i, *_oracle_masked(V[:12_000], Q, 50, labels[:12_000], masks, W, DIMS))


def test_graph_search_with_label_mask(X, one_space):
    V, Q, labels, store = one_space
    q = torch.from_numpy(Q[:60])
    gs = X.engine.GraphSearch(store, 60, 100, with_label_mask=True)
    rng = np.random.default_rng(31)
    for masks in (_masks(60, rng), np.full(60, _bits([3, 9]), dtype=np.int64), None):
        s, i = gs(q, label_mask=masks)
        e_s, e_i = store.search(q, 100, label_mask=masks if masks is not None else -1)
        assert torch.equal(i, e_i) and torch.equal(s, e_s)
    store.set_labels([5], [int(labels[5])])                       # same label, but the label state changed
    with pytest.raises(RuntimeError, match="set_labels"):
        gs(q, label_mask=-1)


def test_labelled_store_unfiltered_equals_unlabelled(X, one_space):
    V, Q, labels, store = one_space
    plain = X.engine.CorpusStore(len(V), (V.shape[1],)).add(torch.from_numpy(V))
    q = torch.from_numpy(Q[:300])
    a_s, a_i = store.search(q, 100)
    b_s, b_i = plain.search(q, 100)
    assert torch.equal(a_i, b_i) and torch.equal(a_s, b_s)
    assert plain.labels is None                                  # never labelled: no label plane


def test_label_validation_and_unsupported_paths(X, one_space):
    V, Q, labels, store = one_space
    with pytest.raises(ValueError):
        store.set_labels([0, 1], [3, 64])
    with pytest.raises(ValueError):
        X.engine.CorpusStore(4, (V.shape[1],)).add(torch.from_numpy(V[:2]), labels=[-1, 0])
    q = torch.from_numpy(Q[:4])
    with pytest.raises(ValueError):
        X.engine.rank_of_gt(store, q, [0, 1, 1, 1, 1], [0], label_mask=-1)
    with pytest.raises(ValueError):
        X.engine.search_norm_score(store, q, 10, label_mask=-1)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_filtered_sharded_search_over_nccl_equals_one_store():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("one visible GPU: the NCCL path needs at least two")
    ranks = min(4, n)
    env = dict(os.environ)
    env.pop("OMP_NUM_THREADS", None)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(ranks),
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tools", "check_filtered_sharded.py")]
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    sys.stdout.write(out.stdout[-4000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "filtered sharded search on %d GPUs: OK" % ranks in out.stdout


def test_short_list_certificate_keeps_tie_cuts(X):
    """600 queries (selection sort of max(2048, 4k) entries per row) whose mask allows only 3 000 identical rows:
    they fit the candidate lists (thr = -inf) but not the sort, so the selection flags them and the re-run with the
    full sort returns the lowest indices of the tie -- the thr = -inf fix-up must not certify such a row."""
    nv, d, nq, k = 60_000, 64, 600, 100
    V, Q = X.synth.gaussian(41, nv, d), X.synth.gaussian(42, nq, d)
    rng = np.random.default_rng(43)
    labels = rng.integers(0, 63, nv).astype(np.uint8)
    tie = np.sort(rng.choice(nv, 3_000, replace=False))
    V[tie] = V[tie[0]]
    labels[tie] = 63
    masks = np.where(np.arange(nq) % 2 == 0, _bits(range(63)), _bits([63])).astype(np.int64)
    store = X.engine.CorpusStore(nv, (d,)).add(torch.from_numpy(V), labels=labels)
    stats = {}
    s, i = store.search(torch.from_numpy(Q), k, label_mask=masks, stats=stats)
    assert stats["thr_inf_rows"] == nq // 2
    ref_i, ref_s = _oracle_masked(V, Q, k, labels, masks)
    # odd rows: the tie, from the one distinct vector (exact ties whatever the BLAS does) -- the k lowest row ids
    tie_s = -linas.cal_error(V[tie[:1]].astype(np.float64), Q[1::2].astype(np.float64))
    ref_i[1::2], ref_s[1::2] = tie[:k], np.broadcast_to(tie_s, (nq // 2, k))
    _assert_oracle(s, i, ref_i, ref_s)
