"""Property tests (hypothesis) of the host-side logic against the oracle restatement.  CPU only."""
import math

from hypothesis import given, settings, strategies as st

from cross_modal_video_engine_b200 import distributed, engine, metrics
from oracle import linas


@settings(max_examples=60, deadline=None)
@given(st.lists(st.integers(0, 12), min_size=0, max_size=25), st.lists(st.tuples(st.integers(0, 14), st.integers(0, 3)),
                                                                     min_size=0, max_size=60))
def test_get_gt_matches_the_reference_loop(video_nums, caps):
    """Duplicated video ids, captions of unknown videos, videos without captions: same containers, same order."""
    video_ids = ["video%d" % v for v in video_nums]
    caption_ids = ["video%d#enc#%d" % (v, c) for v, c in caps]
    v2t, t2v = metrics.get_gt(video_ids, caption_ids)
    v2t_ref, t2v_ref = linas.get_gt(video_ids, caption_ids)
    assert v2t == v2t_ref
    assert t2v == t2v_ref and list(t2v) == list(t2v_ref)


@settings(max_examples=100, deadline=None)
@given(st.integers(0, 10 ** 7), st.integers(1, 16))
def test_shard_ranges_partition_the_rows(n, world):
    spans = [distributed.shard_range(n, world, r) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(spans[:-1], spans[1:]))
    sizes = [hi - lo for lo, hi in spans]
    assert max(sizes) - min(sizes) <= 1


@settings(max_examples=100, deadline=None)
@given(st.integers(1, 1001), st.integers(16385, 2 * 10 ** 7))
def test_plan_invariants(k, n):
    p = engine.plan(k, n)
    assert p["step"] >= 1 and p["n_sample"] == (n + p["step"] - 1) // p["step"]
    assert 1 <= p["j"] <= p["j_cap"] <= p["n_sample"]
    assert 2048 <= p["cap"] <= 32768
    assert p["j"] >= k / p["step"]                       # the order statistic sits above the expected k-th sample
    lam = k / p["step"]
    assert p["margin"] == engine.thr_margin(lam) and p["margin"] in (0.0, 1.0, 2.0)
    # the eps margin may only be dropped while the rank ratio j / lam leaves a score gap of its own
    assert p["margin"] > 0.0 or p["j"] / lam >= 3.3


def test_benchmark_configs_search_without_the_margin():
    """The BASELINE configs keep the margin-free threshold (their candidate counts and result digests are those of
    the committed profiles); deep lists over small corpora get the margin back."""
    for k, n in ((100, 10_000_000), (101, 1_000_000), (1000, 1_080_000), (100, 1_250_000)):
        assert engine.plan(k, n)["margin"] == 0.0
    assert engine.plan(1000, 200_000)["margin"] == 1.0
    assert engine.plan(8000, 20_000)["margin"] == 2.0


@settings(max_examples=100, deadline=None)
@given(st.floats(1e-5, 4e-3), st.floats(1e-5, 4e-3), st.lists(st.floats(0.05, 2.0), min_size=1, max_size=4),
       st.integers(64, 8192))
def test_measured_eps_is_monotone_and_covers_the_cauchy_schwarz_terms(dq, dv, wts, k_len):
    e = engine.measured_eps(dq, dv, wts, len(wts), k_len)
    qn = math.sqrt(sum(w * w for w in wts))
    assert e >= dq * math.sqrt(len(wts)) + qn * dv        # operand rounding, both sides
    assert engine.measured_eps(dq * 1.5, dv, wts, len(wts), k_len) > e
    assert engine.measured_eps(dq, dv * 1.5, wts, len(wts), k_len) > e
    assert engine.measured_eps(dq, dv, wts, len(wts), 2 * k_len) > e


def _apriori_bound(wts, dims):
    """|bf16-operand score - exact score| without measured residuals: each space's product moves by at most
    |w_s| (2u + u^2) under rounding to bf16 (u = 2^-8), the fp32 accumulation of K products by at most
    K 2^-22 |Qb| |Vb| with |Qb| <= |w| (1 + u), |Vb| <= sqrt(S) (1 + u), plus 1e-6 for the fp32 rounding of the operand."""
    u = 2.0 ** -8
    k_len = sum(-(-d // 64) * 64 for d in dims)
    w_norm = math.sqrt(sum(w * w for w in wts))
    return (sum(abs(w) for w in wts) * (2 * u + u * u)
            + k_len * 2.0 ** -22 * w_norm * (1 + u) * math.sqrt(len(dims)) * (1 + u) + 1e-6), k_len


@settings(max_examples=300, deadline=None)
@given(st.lists(st.tuples(st.integers(1, 6000), st.floats(0.05, 2.0), st.booleans()), min_size=1, max_size=4)
       .filter(lambda sp: sum(d for d, _, _ in sp) <= 6000))
def test_fallback_eps_covers_the_a_priori_bound(spaces):
    """A NaN residual (a zero row under 'plain') makes eps the fallback bound: it must cover the a-priori bound for every
    layout the store accepts (up to 6000 raw columns), whatever K, and reach the device as a float without rounding
    down.  Where 8.5e-3 per unit weight already covered it, the fallback stays that constant."""
    import numpy as np
    dims = [d for d, _, _ in spaces]
    wts = [-w if neg else w for _, w, neg in spaces]
    bound, k_len = _apriori_bound(wts, dims)
    e = engine.measured_eps(float("nan"), 1e-3, wts, len(dims), k_len)
    assert e >= bound
    assert e <= max(bound, engine.EPS_X1 * max(1.0, sum(abs(w) for w in wts))) * (1 + 1e-6)
    assert float(np.float32(e)) == e


def test_fallback_eps_for_long_rows():
    """The layouts where a constant 8.5e-3 per unit weight fell below the bound."""
    for dims, wts in (((2048,), (1.0,)), ((2816,), (1.0,)), ((6000,), (1.0,)), ((3000, 3000), (1.0, 1.0)),
                      ((3000, 2000), (0.5, 0.5)), ((1536, 512), (0.6, -0.4))):
        bound, k_len = _apriori_bound(wts, dims)
        assert engine.measured_eps(float("nan"), float("nan"), wts, len(dims), k_len) >= bound, (dims, wts)
