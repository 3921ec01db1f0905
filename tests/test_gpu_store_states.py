"""Search and ground-truth ranks on stores in the states the public API allows besides "created at its final size and
filled once" (B200 only): filled below capacity, grown between searches, a captured GraphSearch after growth, a
head-stream search issued straight after an ``add``, and float-tied exact scores beyond the selection's sort
capacity with 512 queries or more.  Every result is compared with the fp64 oracle (``oracle/linas.py``): indices
exactly, scores within 1e-13."""
import numpy as np
import pytest
import torch

from oracle import linas
from test_gpu_parity import _oracle_topk

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def X():
    from cross_modal_video_engine_b200 import _native, engine, metrics, synth
    _native.require_device()

    class NS:
        pass
    ns = NS()
    ns.__dict__.update(dict(native=_native, engine=engine, metrics=metrics, synth=synth))
    return ns


DIMS, W = (96, 32), (0.7, 0.3)


@pytest.fixture(scope="module")
def planted():
    """40 000 two-space videos and 300 captions, caption j planted near video j (all in the first 25 000 rows)."""
    from cross_modal_video_engine_b200 import synth
    V, Q, vid, cap, _ = synth.msrvtt_like(19, 40_000, 1, sum(DIMS), 2.5)
    return V, Q[:300], vid, cap[:300]


def _fused(V, Q):
    V64, Q64 = V.astype(np.float64), Q.astype(np.float64)
    return linas.fused_errors([V64[:, :DIMS[0]], V64[:, DIMS[0]:]], [Q64[:, :DIMS[0]], Q64[:, DIMS[0]:]], W)


def _assert_oracle(s, i, ref_idx, ref_s):
    np.testing.assert_array_equal(i.cpu().numpy(), ref_idx)
    np.testing.assert_allclose(s.cpu().numpy(), ref_s, rtol=0, atol=1e-13)


def test_partially_filled_store_then_grown(X, planted):
    """A two-space store of capacity 60 000 filled with 25 000 rows in two ragged adds: the norm planes are
    [S, capacity], so the exact rescore of space 1 must find its norms one capacity (not one row count) further on.
    Searches (with and without exclusions), exact ground-truth ranks and eval_q2m equal the oracle's; after 15 000
    more rows the search covers all 40 000 and equals a store filled once."""
    V, Q, vid, cap = planted
    k, n1 = 100, 25_000
    store = X.engine.CorpusStore(60_000, DIMS)
    store.add(torch.from_numpy(V[:11_000])).add(torch.from_numpy(V[11_000:n1]))
    s, i = store.search(torch.from_numpy(Q), k, weights=W)
    _assert_oracle(s, i, *_oracle_topk(V[:n1], Q, k, weights=W, dims=DIMS))
    excl = np.arange(len(Q))                                     # each caption's own video (rank 1 for most)
    s, i = store.search(torch.from_numpy(Q), k, weights=W, exclude=excl)
    _assert_oracle(s, i, *_oracle_topk(V[:n1], Q, k, weights=W, dims=DIMS, exclude=excl))
    # exact ranks of the planted ground truths without the matrix
    _, t2v_gt = linas.get_gt(vid[:n1], cap)
    err = _fused(V[:n1], Q)
    ref = linas.eval_q2m(err, t2v_gt)
    res = X.metrics.RankResult.from_store(store, torch.from_numpy(Q), t2v_gt, weights=W, first_only=True)
    np.testing.assert_array_equal(res.ranks.cpu().numpy(), linas.gt_ranks(err, t2v_gt))
    assert res.recall_medr_meanr() == ref and 2.0 < ref[0] < 98.0 and ref[4] > 10.0       # non-degenerate
    assert X.metrics.eval_q2m_store(store, torch.from_numpy(Q), t2v_gt, weights=W) == ref
    # grow the store: the cached residual maximum follows the row count
    store.add(torch.from_numpy(V[n1:]))
    s, i = store.search(torch.from_numpy(Q), k, weights=W)
    _assert_oracle(s, i, *_oracle_topk(V, Q, k, weights=W, dims=DIMS))
    full = X.engine.CorpusStore(len(V), DIMS).add(torch.from_numpy(V))
    s_f, i_f = full.search(torch.from_numpy(Q), k, weights=W)
    assert torch.equal(i, i_f) and torch.equal(s, s_f)
    want = float(store.resid[:, :store.n].sum(0).max())
    assert float(store.resid_max2()) == want
    assert float(X.engine._dv2_global([store], X.engine.SoloComm())) == want


@pytest.fixture(scope="module", params=["copies", "nudged"])
def tied(request):
    """40 000 x 64 corpus in which 3 000 rows are copies of one vector u (2 700 in rows [0, 20 000), 300 in
    [20 000, 40 000)), and 600 queries u + 0.1 noise: the copies are every query's top 3 000.

    ``copies``: exact ties; the top-100 are the 100 smallest copies.  ``nudged``: one coordinate of each copy moved
    up by 0-31 float steps, so the fp64 scores take 32 distinct values (> 1e-12 apart) that still agree to float
    precision: the top-100 are the best one or two levels, rows from all over the corpus, so a list that keeps an
    arbitrary subset of the float ties misses some of them."""
    rng = np.random.default_rng(77)
    n, d, nq, k = 40_000, 64, 600, 100
    V = rng.standard_normal((n, d)).astype(np.float32)
    u = rng.standard_normal(d).astype(np.float32)
    dup = np.sort(np.concatenate([rng.choice(20_000, 2_700, replace=False),
                                  20_000 + rng.choice(20_000, 300, replace=False)]))
    V[dup] = u
    Q = (u + 0.1 * rng.standard_normal((nq, d))).astype(np.float32)
    if request.param == "nudged":
        c = int(np.argmax(np.abs(u)))
        V[dup, c] = u[c] + rng.integers(0, 32, len(dup)).astype(np.float32) * np.spacing(np.abs(u[c]))
    # reference from the UNIQUE vectors, gathered to the copies: the ties are exact whatever the BLAS does
    uniq, inv = np.unique(V, axis=0, return_inverse=True)
    err = linas.cal_error(uniq.astype(np.float64), Q.astype(np.float64))[:, inv.reshape(-1)]
    ref_idx = np.argsort(err, axis=1, kind="stable")[:, :k]
    ref_s = -np.take_along_axis(err, ref_idx, axis=1)
    if request.param == "copies":
        assert (ref_idx == dup[:k][None, :]).all()              # the top-100 are the 100 smallest copies ...
        assert (ref_s == ref_s[:, :1]).all()                    # ... and their scores really are tied
    else:
        kth = ref_s[:, -1:].astype(np.float32)
        assert (((-err[:, :20_000]).astype(np.float32) == kth).sum(1) > 2048).mean() > 0.8   # float ties in shard 0
        top = -np.sort(err, axis=1)[:, :k + 1]
        assert min(np.diff(np.unique(r)).min() for r in top if len(np.unique(r)) > 1) > 1e-12  # order is robust
        assert (np.searchsorted(dup, ref_idx) >= 2048).any(axis=1).all()   # beyond the first 2 048 copies
    return V, Q, k, ref_idx, ref_s


def test_heavy_ties_many_queries_one_store(X, tied):
    """600 queries whose top 3 000 are float-tied: more than the 2 048 entries the selection sorts per row when 512
    rows or more are selected at once.  The re-run must select in smaller batches and certify the exact list (not
    give up with an XmveError)."""
    V, Q, k, ref_idx, ref_s = tied
    store = X.engine.CorpusStore(len(V), (V.shape[1],)).add(torch.from_numpy(V))
    s, i = store.search(torch.from_numpy(Q), k)
    _assert_oracle(s, i, ref_idx, ref_s)


def test_heavy_ties_many_queries_two_shards(X, tied):
    """The same over two stores on one GPU (packed lists + merge): the shard holding 2 700 copies cannot sort them all
    in a 600-row selection and must flag its list, so that the merge does not certify an arbitrary subset (with
    ``nudged`` such a subset misses part of the top-100; with exact copies it may happen to hold the smallest rows)."""
    V, Q, k, ref_idx, ref_s = tied
    cut = 20_000
    shards = [X.engine.CorpusStore(cut, (V.shape[1],)).add(torch.from_numpy(V[:cut])),
              X.engine.CorpusStore(len(V) - cut, (V.shape[1],), index_offset=cut).add(torch.from_numpy(V[cut:]))]
    s, i = X.engine.search_shards(shards, torch.from_numpy(Q), k)
    _assert_oracle(s, i, ref_idx, ref_s)


def test_graph_search_refuses_a_grown_store(X):
    """A GraphSearch captured over 60 000 rows of a 120 000-row store; 60 000 more rows arrive, each query's
    near-duplicate among them.  A replay would search the old rows only: it must raise instead, and a new capture
    finds every planted row."""
    nv, d, nq, k = 60_000, 128, 48, 20
    V = X.synth.gaussian(66, 2 * nv, d)
    Q = X.synth.gaussian(67, nq, d)
    plant = nv + np.random.default_rng(68).choice(nv, nq, replace=False)
    V[plant] = 2.0 * Q + 0.05 * X.synth.gaussian(69, nq, d)
    store = X.engine.CorpusStore(2 * nv, (d,)).add(torch.from_numpy(V[:nv]))
    gs = X.engine.GraphSearch(store, nq, k)
    s0, i0 = gs(torch.from_numpy(Q))
    _assert_oracle(s0, i0, *_oracle_topk(V[:nv], Q, k))
    store.add(torch.from_numpy(V[nv:]))
    with pytest.raises(RuntimeError, match="corpus changed"):
        gs(torch.from_numpy(Q))
    ref_idx, ref_s = _oracle_topk(V, Q, k)
    assert (ref_idx[:, 0] == plant).all()
    s, i = X.engine.GraphSearch(store, nq, k)(torch.from_numpy(Q))
    _assert_oracle(s, i, ref_idx, ref_s)


def test_head_stream_search_straight_after_add(X, planted):
    """search_shards(head_stream=h) right after ``add`` while the add's K1 is still queued (behind a bounded ~50 ms
    spin on the current stream): the head reduces the corpus residuals and samples the operand, so it must wait for
    the add.  Otherwise it measures zero residuals, caches that bound for the corpus state, and every later search
    uses an eps that is no bound."""
    V, Q, _, _ = planted
    k = 50
    store = X.engine.CorpusStore(len(V), DIMS)
    V_dev, Q_dev = torch.from_numpy(V).cuda(), torch.from_numpy(Q).cuda()
    head = torch.cuda.Stream()
    torch.cuda.synchronize()
    torch.cuda._sleep(100_000_000)                              # K1 of the add queues behind this spin
    store.add(V_dev)
    s, i = X.engine.search_shards([store], Q_dev, k, weights=W, defer=True, head_stream=head).result()
    torch.cuda.synchronize()
    dv2 = float(X.engine._dv2_global([store], X.engine.SoloComm()))                   # the cached value
    assert dv2 == float(store.resid[:, :store.n].sum(0).max()) and dv2 > 0.0
    s_e, i_e = store.search(Q_dev, k, weights=W)
    assert torch.equal(i, i_e) and torch.equal(s, s_e)
    _assert_oracle(s, i, *_oracle_topk(V, Q, k, weights=W, dims=DIMS))
