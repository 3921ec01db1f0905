"""Similar pairs on the B200: ``xmve_pair_select`` against a torch statement, and ``similar_pairs`` against the fp64
oracle (``oracle.linas``) and a torch fp64 statement computed on the device: for every row i the list is exactly
``{j > i : S[i, j] >= t}``, scores within 1e-12, ordered by (score desc, j asc).  Tests that need several blocks
lower ``engine.PAIR_BLOCK`` so that blocks break inside groups of duplicates.  Also: consistency with
``range_search``, two stores against one, the edges, the sized ``MemoryError``, ``cli.py pairs`` and the NCCL path on
two GPUs or more."""
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
    """torch statement of the order: (score desc, row asc) per row of [rows, n]."""
    o = torch.argsort(i, dim=1, stable=True)
    s, i = torch.gather(s, 1, o), torch.gather(i, 1, o)
    o = torch.argsort(s, dim=1, descending=True, stable=True)
    return torch.gather(s, 1, o), torch.gather(i, 1, o)


def _store(X, V, dims, capacity=None):
    st = X.engine.CorpusStore(capacity or max(len(V), 1), dims)
    if len(V):
        st.add(torch.as_tensor(V))
    return st


# ---- kernel -------------------------------------------------------------------------------------------------------
def _select(X, exact, cand_idx, counts, idx_offset, ms, after):
    """count + cumsum + fill through the engine helper -> (counts, offsets, scores, idx)."""
    cand = (counts, None, cand_idx)
    kw = {} if after is None else {"after": after}
    cnt = X.engine._range_select(exact, cand, idx_offset, None, ms, **kw)
    off = torch.zeros(len(cnt) + 1, dtype=torch.int64, device="cuda")
    off[1:] = torch.cumsum(cnt, 0)
    out_s = torch.empty(int(off[-1]), dtype=torch.float64, device="cuda")
    out_i = torch.empty(int(off[-1]), dtype=torch.int64, device="cuda")
    X.engine._range_select(exact, cand, idx_offset, None, ms, counts=cnt, off=off[:-1],
                           max_len=min(exact.shape[1], int(cnt.max())), out_s=out_s, out_i=out_i, **kw)
    torch.cuda.synchronize()
    return cnt, off, out_s, out_i


def test_pair_select_kernel(X):
    rows, cap, off0 = 600, 40960, 1000
    g = torch.Generator(device="cuda").manual_seed(7)
    exact = torch.rand((rows, cap), generator=g, device="cuda", dtype=torch.float64)
    cand_idx = torch.argsort(torch.rand((rows, cap), generator=g, device="cuda"), dim=1).to(torch.int32) * 3
    counts = torch.randint(0, 400, (rows,), generator=g, device="cuda", dtype=torch.int32)
    ms = torch.full((rows,), 0.3, dtype=torch.float64, device="cuda")
    ids = cand_idx.long() + off0
    # floors that cut every row in the middle of its listed rows
    after = torch.tensor([int(ids[r, :max(1, int(counts[r]))].median()) for r in range(rows)], device="cuda")
    after[0] = -1                                                  # the range_select result
    after[1] = 1 << 40                                             # above every row: nothing
    counts[2], ms[2], after[2] = 40000, -INF, off0 + 3 * 4000     # ~36 000 matches: the scratch path
    counts[3], ms[3], after[3] = 20000, -INF, off0 + 3 * 40000    # a high floor: a few hundred matches
    exact[4, :300] = torch.round(exact[4, :300] * 8) / 8           # ties at the minimum, ordered by row
    counts[4], ms[4], after[4] = 300, 0.5, int(ids[4, :300].median())
    exact[5, :100] = float("nan")                                  # NaN never matches
    exact[6, :300] = -INF                                          # -inf never matches, even for -inf
    ms[6] = -INF
    counts[7] = cap + 50                                           # an overflowed list: only cap entries are read
    cnt, off, out_s, out_i = _select(X, exact, cand_idx, counts, off0, ms, after)
    n = torch.minimum(counts.long(), torch.tensor(cap, device="cuda"))
    hit = (torch.arange(cap, device="cuda")[None, :] < n[:, None]) & (exact > -INF) & (exact >= ms[:, None]) \
        & (ids > after[:, None])
    assert torch.equal(cnt, hit.sum(1))
    assert int(cnt[1]) == 0 and int(cnt[2]) > 16384 and 0 < int(cnt[4]) < int(((exact[4, :300] >= 0.5)).sum())
    listed = (torch.arange(cap, device="cuda")[None, :] < n[:, None]) & (exact >= ms[:, None])
    assert 0 < int(cnt[8:].sum()) < int(listed[8:].sum())           # the floors cut the rows
    ws, wi = _sorted_pairs(torch.where(hit, exact, torch.full_like(exact, -INF)),
                           torch.where(hit, ids, torch.full_like(ids, 1 << 62)))
    keep = torch.arange(cap, device="cuda")[None, :] < cnt[:, None]
    assert torch.equal(out_i, wi[keep]) and torch.equal(out_s, ws[keep])
    # after = -1 everywhere: xmve_range_select's result
    r_cnt, r_off, r_s, r_i = _select(X, exact, cand_idx, counts, off0, ms, None)
    p_cnt, p_off, p_s, p_i = _select(X, exact, cand_idx, counts, off0, ms, torch.full_like(after, -1))
    assert torch.equal(r_cnt, p_cnt) and torch.equal(r_i, p_i) and torch.equal(r_s, p_s)


# ---- against the fp64 oracle ----------------------------------------------------------------------------------------
def _oracle_pairs_scores(V, dims=None, weights=None):
    V64 = V.astype(np.float64)
    if dims is None:
        return -linas.cal_error(V64, V64)
    offs = np.cumsum((0,) + tuple(dims))
    sp = [V64[:, a:b] for a, b in zip(offs[:-1], offs[1:])]
    return -linas.fused_errors(sp, sp, weights)


def _check_oracle(res, S, t):
    n = len(S)
    off = res.offsets.cpu().numpy()
    scores, idx = res.scores.cpu().numpy(), res.idx.cpu().numpy()
    assert len(off) == n + 1 and off[0] == 0 and off[-1] == len(idx)
    for i in range(n):
        want = np.nonzero(S[i, i + 1:] >= t)[0] + i + 1
        s, j = scores[off[i]:off[i + 1]], idx[off[i]:off[i + 1]]
        np.testing.assert_array_equal(np.sort(j), want, err_msg="row %d" % i)
        np.testing.assert_allclose(s, S[i, j], rtol=0, atol=1e-12)
        assert np.all((s[:-1] > s[1:]) | ((s[:-1] == s[1:]) & (j[:-1] < j[1:]))), "row %d is not sorted" % i


@pytest.mark.parametrize("spaces", ["one", "two"])
def test_similar_pairs_match_oracle(X, monkeypatch, spaces):
    monkeypatch.setattr(X.engine, "PAIR_BLOCK", 256)
    dims, w = ((160,), None) if spaces == "one" else ((128, 64), (0.6, 0.4))
    V = X.synth.clustered(11, 2000, sum(dims))
    V[700:720] = V[690]                                            # exact copies across a block boundary (768)
    V[760:780] = V[5]
    S = _oracle_pairs_scores(V, None if spaces == "one" else dims, w)
    up = np.sort(S[np.triu_indices(len(V), 1)])[::-1]
    j = 20000
    while up[j - 1] - up[j] < 1e-9:
        j += 1
    t = 0.5 * (up[j - 1] + up[j])
    stats = {}
    res = _store(X, V, dims).similar_pairs(t, weights=w, stats=stats)
    _check_oracle(res, S, t)
    assert stats["pairs"] == res.idx.numel() >= 20000 and stats["blocks"] == 8 and 0 < stats["eps"] < X.engine.EPS_X1


def test_similar_pairs_all_and_none(X):
    V = X.synth.clustered(21, 300, 64)
    store = _store(X, V, (64,))
    S = _oracle_pairs_scores(V)
    res = store.similar_pairs(-INF)
    assert res.idx.numel() == 300 * 299 // 2 == 44850
    _check_oracle(res, S, -INF)
    res = store.similar_pairs(INF)
    assert res.idx.numel() == 0 and torch.equal(res.offsets, torch.zeros(301, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError, match="NaN"):
        store.similar_pairs(float("nan"))
    empty = X.engine.CorpusStore(16, (64,))
    res = empty.similar_pairs(0.5)
    assert res.offsets.tolist() == [0] and res.idx.numel() == 0
    one = _store(X, V[:1], (64,))
    res = one.similar_pairs(-INF)
    assert res.offsets.tolist() == [0, 0] and res.scores.numel() == 0
    # rows that no shard holds (a store whose first global row is 100) get empty lists
    late = X.engine.CorpusStore(300, (64,), index_offset=100).add(torch.from_numpy(V))
    res = late.similar_pairs(-INF)
    assert res.offsets.numel() == 401 and int(res.offsets[100]) == 0 and res.idx.numel() == 44850
    assert int(res.idx.min()) == 101


# ---- a larger store against a torch fp64 statement on the device --------------------------------------------------
DIMS, W, T = (128, 64), (0.6, 0.4), 0.9


def _planted(n, seed):
    """Gaussian rows with planted near-copies (cosine about 0.95 - 0.99) and groups of exact copies: one group of
    2 100 copies (its lists overflow the first pass), one across the block boundary at row 1024 and small groups."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    V = torch.randn((n, sum(DIMS)), generator=g, device="cuda")
    for j in range(50, n, 50):
        src = int(torch.randint(0, j, (1,), generator=g, device="cuda"))
        sigma = 0.15 + 0.18 * float(torch.rand((), generator=g, device="cuda"))
        V[j] = V[src] + sigma * torch.randn((sum(DIMS),), generator=g, device="cuda")
    for k in range(20):
        rows = torch.randint(0, n, (5,), generator=g, device="cuda")
        V[rows] = V[rows[0]].clone()
    V[1015:1035] = V[1015].clone()
    V[torch.arange(10001, 10001 + 2100 * 23, 23, device="cuda")] = V[3].clone()     # last: the group stays whole
    return V


def _unit(V):
    out, o = [], 0
    for d in DIMS:
        x = V[:, o:o + d].double()
        out.append(x / torch.linalg.vector_norm(x, dim=1, keepdim=True))
        o += d
    return out


def _check_statement(res, V, t, blk=4096):
    n = len(V)
    U = _unit(V)
    off = res.offsets
    assert off.numel() == n + 1 and int(off[-1]) == res.idx.numel()
    lens = off[1:] - off[:-1]
    row = torch.repeat_interleave(torch.arange(n, device="cuda"), lens)
    s, j = res.scores, res.idx
    same = row[1:] == row[:-1]
    assert bool((~same | (s[:-1] > s[1:]) | ((s[:-1] == s[1:]) & (j[:-1] < j[1:]))).all()), "lists are not sorted"
    cols = torch.arange(n, device="cuda")
    for b0 in range(0, n, blk):
        b1 = min(n, b0 + blk)
        S = sum(w * (u[b0:b1] @ u.T) for w, u in zip(W, U))
        upper = cols[None, :] > torch.arange(b0, b1, device="cuda")[:, None]
        assert not bool((upper & ((S - t).abs() < 1e-10)).any()), "a score within 1e-10 of the minimum"
        want = upper & (S >= t)
        assert torch.equal(lens[b0:b1], want.sum(1))
        e0, e1 = int(off[b0]), int(off[b1])
        key = (row[e0:e1] - b0) * n + j[e0:e1]
        o = torch.argsort(key)
        wr, wj = torch.nonzero(want, as_tuple=True)
        assert torch.equal(key[o], wr * n + wj)
        assert bool(((s[e0:e1][o] - S[wr, wj]).abs() <= 1e-12).all())


@pytest.fixture(scope="module")
def planted(X):
    """60 000 planted rows in a store of capacity 64 000 grown by two adds, and its pairs at PAIR_BLOCK = 512."""
    V = _planted(60000, 31)
    store = X.engine.CorpusStore(64000, DIMS)
    store.add(V[:31111])
    store.add(V[31111:])
    old = X.engine.PAIR_BLOCK
    X.engine.PAIR_BLOCK = 512
    try:
        stats = {}
        res = store.similar_pairs(T, weights=W, stats=stats)
    finally:
        X.engine.PAIR_BLOCK = old
    return V, store, res, stats


def test_similar_pairs_planted_store(X, planted):
    V, store, res, stats = planted
    _check_statement(res, V, T)
    assert res.idx.numel() > 2100 * 2099 // 2 and stats["rerun_rows"] > 0 and stats["blocks"] == 118
    # the exact copies of row 3 pair with each other, once per pair
    grp = torch.cat([torch.tensor([3], device="cuda"), torch.arange(10001, 10001 + 2100 * 23, 23, device="cuda")])
    i, j, s = res.pairs()
    inside = torch.isin(i, grp) & torch.isin(j, grp)
    assert int(inside.sum()) == 2101 * 2100 // 2 and bool((i < j).all())


def test_similar_pairs_equal_range_search(X, planted):
    """Row i's list is the j > i part of range_search(V[i]), with bit-identical scores."""
    V, store, res, _ = planted
    g = torch.Generator().manual_seed(3)
    rows = torch.cat([torch.tensor([3, 1015, 1023, 1024, 10001, 59999]), torch.randint(0, 60000, (40,), generator=g)])
    for i in rows.tolist():
        r = store.range_search(V[i:i + 1], T, weights=W)
        keep = r.idx > i
        a, b = int(res.offsets[i]), int(res.offsets[i + 1])
        assert torch.equal(res.idx[a:b], r.idx[keep]) and torch.equal(res.scores[a:b], r.scores[keep]), "row %d" % i


def test_two_stores_equal_one(X, monkeypatch, planted):
    monkeypatch.setattr(X.engine, "PAIR_BLOCK", 512)
    V = planted[0][:36000]
    one = _store(X, V, DIMS)
    a = X.engine.CorpusStore(20000, DIMS, index_offset=0).add(V[:20000])        # 20 000 is not a multiple of 512
    b = X.engine.CorpusStore(16000, DIMS, index_offset=20000).add(V[20000:])
    r1 = one.similar_pairs(T, weights=W)
    r2 = X.engine.similar_pairs_shards([a, b], T, weights=W)
    assert r1.idx.numel() > 0
    assert torch.equal(r1.offsets, r2.offsets) and torch.equal(r1.idx, r2.idx) and torch.equal(r1.scores, r2.scores)


def test_similar_pairs_refuses_an_output_that_cannot_fit(X):
    """min_score = -inf over 400 000 rows: the first block alone lists 3.3e9 pairs.  The call raises a sized
    MemoryError before it allocates them."""
    V = X.synth.device_gaussian(400000, 64, 5, "cuda")
    store = _store(X, V, (64,))
    torch.cuda.reset_peak_memory_stats()
    with pytest.raises(MemoryError, match="raise min_score"):
        store.similar_pairs(-INF)
    assert torch.cuda.max_memory_allocated() < 40e9


def test_cli_pairs(X, tmp_path, capsys):
    from cross_modal_video_engine_b200 import cli, corpus_io
    V = X.synth.gaussian(41, 400, 64)
    V[[120, 300]] = V[10]                                          # exact copies
    V[350] = V[20] + 0.1 * X.synth.gaussian(42, 1, 64)[0]          # a near-copy
    vid = ["video%d" % i for i in range(len(V))]
    corpus_io.write_bigfile(str(tmp_path / "bf"), vid, V)
    S = _oracle_pairs_scores(V)
    want = [(vid[i], vid[j]) for i in range(len(V)) for j in range(i + 1, len(V)) if S[i, j] >= 0.95]
    assert ("video10", "video120") in want and ("video20", "video350") in want and len(want) == 4
    assert cli.main(["pairs", "--corpus", str(tmp_path / "bf"), "--min-score", "0.95"]) == 0
    lines = [ln.split() for ln in capsys.readouterr().out.strip().splitlines()]
    assert sorted((a, b) for a, b, _ in lines) == sorted(want)
    assert all(abs(float(s) - S[vid.index(a), vid.index(b)]) < 1e-12 for a, b, s in lines)
    out = tmp_path / "pairs.txt"
    assert cli.main(["pairs", "--corpus", str(tmp_path / "bf"), "--min-score", "0.95", "--out", str(out)]) == 0
    assert [ln.split() for ln in out.read_text().splitlines()] == lines


# ---- several GPUs (NCCL) ------------------------------------------------------------------------------------------
def test_similar_pairs_nccl():
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs two GPUs or more")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc_per_node", str(min(4, n)),
                          "--master_port", str(port), os.path.join(ROOT, "tools", "check_pairs_sharded.py")],
                         cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "pairs sharded ok" in out.stdout
