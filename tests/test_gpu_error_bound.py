"""The error bound eps against the B200 (B200 only).

Every exact answer rests on ``|tensor-core score - exact fp64 score| <= eps`` (DESIGN section 5): the top-k
certificate, the pilot bound, range-search completeness, ``rank_of_gt`` bands and similar-pairs thresholds.  eps comes
from K1's measured bf16 residuals.  These tests confront that inequality with the hardware:

1. K1's residual is an upper bound of the operand's real rounding error, on every path ``xmve_prepare_rows`` takes.
2. eps bounds every score of every tile of ``xmve_score_store`` and ``xmve_score_filter``, on data built to make the
   rounding errors add up (coherent rounding), to cancel large partial sums, or to put the norm in one component.
   The fp32 accumulation term ``K 2^-22 |Qb| |Vb|`` is checked on its own against the fp64 product of the operands.
3. Searches stay exact when about 2 000 rows per query have exact scores within eps / 8 of the answer's boundary.

The oracle is a torch fp64 statement over the raw fp32 rows, regenerated from the seed (DESIGN section 2); the
buffers K1 wrote enter only as the quantities under test.  Run with ``-s`` to see the measured ratios."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
U = 2.0 ** -8                                     # bf16 unit roundoff
TILES = (0, 1, 2, 4, 5, 6)


@pytest.fixture(scope="module")
def X():
    from cross_modal_video_engine_b200 import _native, engine
    _native.require_device()

    class NS:
        pass
    ns = NS()
    ns.N, ns.engine = _native, engine
    return ns


def _rup(x, m):
    return (x + m - 1) // m * m


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _pool(x):
    """The frame mean as K1 forms it: fp32 sum over the frames in order, then one fp32 division (by a tensor:
    torch divides by a scalar as a multiplication by its reciprocal)."""
    if x.dim() == 2:
        return x
    s = x[:, 0].clone()
    for f in range(1, x.shape[1]):
        s = s + x[:, f]
    return s / torch.full_like(s, float(x.shape[1]))


def _unit(x64, mode):
    n = torch.linalg.vector_norm(x64, dim=1, keepdim=True)
    return x64 / (n.clamp_min(1e-12) if mode == "eps" else n)


def _exact(q_raw, v_raw, dims, wts, mode):
    """fp64 fused cosine scores [nq, nv] of pooled fp32 rows."""
    out, o = 0.0, 0
    for d, w in zip(dims, wts):
        out = out + w * (_unit(q_raw[:, o:o + d].double(), mode) @ _unit(v_raw[:, o:o + d].double(), mode).T)
        o += d
    return out


# ---- 1. K1's residual ---------------------------------------------------------------------------------------------
def _special_rows(d, g):
    """Rows K1 must get right: plain Gaussian, scaled to 1e30 and 1e-30, a norm below 1e-12, and rows whose
    normalised components are all bf16-exact (one, four and sixteen entries of +-1)."""
    rows = [torch.randn(d, generator=g, device="cuda") for _ in range(6)]
    rows += [torch.randn(d, generator=g, device="cuda") * 1e30, torch.randn(d, generator=g, device="cuda") * 1e-30,
             torch.randn(d, generator=g, device="cuda") * 1e-14]
    for m in (1, 4, 16):
        r = torch.zeros(d, device="cuda")
        pos = torch.randperm(d, generator=g, device="cuda")[:m]
        r[pos] = torch.where(torch.rand(m, generator=g, device="cuda") < 0.5, -1.0, 1.0)
        rows += [r, r * 1e30]
    return torch.stack(rows)


# name, d, frames, dtype, src_ld - frames * d, raw_off, op_off
K1_PATHS = [
    ("fast8", 1024, 1, torch.float32, 0, 0, 0),
    ("fast16", 1028, 1, torch.float32, 0, 4, 64),
    ("fast16", 2048, 1, torch.float32, 4, 0, 0),
    ("generic", 2052, 1, torch.float32, 0, 0, 0),
    ("generic_odd_d", 1001, 1, torch.float32, 0, 0, 0),
    ("generic_src_ld", 1024, 1, torch.float32, 1, 0, 0),
    ("generic_raw_off", 512, 1, torch.float32, 0, 1, 0),
    ("generic_op_off", 512, 1, torch.float32, 0, 0, 2),
    ("f64", 768, 1, torch.float64, 0, 0, 0),
    ("fast_frames", 512, 3, torch.float32, 0, 0, 0),
    ("generic_frames", 513, 2, torch.float32, 0, 0, 0),
]


@pytest.mark.parametrize("weight", [0.6, 1.0, -0.4])
@pytest.mark.parametrize("mode", ["plain", "eps"])
@pytest.mark.parametrize("path", K1_PATHS, ids=lambda p: "%s-%d" % (p[0], p[1]))
def test_k1_residual_bounds_the_operand_rounding(X, path, mode, weight):
    """``sqrt(resid) + 2^-23 |w| >= |w x / den - operand|`` per row (the allowance is the fp32 rounding of ``y``,
    which the 1e-6 term of eps absorbs) and ``resid <= 1.0011 (ref + allowance)``: an upper bound, not a loose one."""
    N = X.N
    name, d, frames, dtype, ld_pad, raw_off, op_off = path
    g = _gen(7 + d)
    base = _special_rows(d, g)
    if mode == "eps":                                       # a zero row is defined under 'eps' only
        base = torch.cat([base, torch.zeros((1, d), device="cuda")])
    n = base.shape[0]
    if frames == 1:
        x = base
    else:                                                   # frames whose fp32 mean is the base row, plus noise
        x = base.unsqueeze(1) * (1 + 0.01 * torch.randn((n, frames, 1), generator=g, device="cuda"))
    x = x.reshape(n, frames * d)
    src = torch.zeros((n, frames * d + ld_pad), dtype=dtype, device="cuda")
    src[:, :frames * d] = x.to(dtype)
    dpad = _rup(d, 64)
    raw = torch.zeros((n, _rup(raw_off + d, 4) + 4), dtype=torch.float32, device="cuda")    # row strides the
    op = torch.zeros((n, _rup(op_off + dpad, 4) + 4), dtype=torch.bfloat16, device="cuda")  # fast path accepts
    nrm = torch.zeros(n, dtype=torch.float64, device="cuda")
    res = torch.zeros(n, dtype=torch.float32, device="cuda")
    N.call("xmve_prepare_rows", N.ptr(src), N.F64 if dtype == torch.float64 else N.F32, n, d, frames, src.stride(0),
           N.ptr(raw), raw.stride(0), raw_off, N.ptr(nrm), N.ptr(res), N.ptr(op), op.stride(0), op_off, N.OP_X1,
           weight, N.NORM_EPS if mode == "eps" else N.NORM_PLAIN, N.stream_ptr())
    torch.cuda.synchronize()
    pooled = _pool(src[:, :frames * d].float().reshape(n, frames, d) if frames > 1 else src[:, :d].float())
    assert torch.equal(raw[:, raw_off:raw_off + d], pooled)
    y = float(np.float32(weight)) * _unit(pooled.double(), mode)   # w x / den in fp64, w as the kernel gets it
    ref = ((y - op[:, op_off:op_off + d].double()) ** 2).sum(1)
    allow = 2.0 ** -23 * abs(weight)
    r = res.double()
    bad = ~(r.sqrt() + allow >= ref.sqrt())
    assert not bad.any(), "%s: residual below the rounding error in rows %s (resid %s, ref %s)" % (
        name, bad.nonzero().flatten().tolist(), r[bad].tolist(), ref[bad].tolist())
    assert torch.all(r <= 1.0011 * (ref.sqrt() + allow) ** 2), name
    assert torch.all(r.sqrt() <= abs(weight) * U * 1.0001)                  # the a-priori worst case per space
    exact_rows = torch.arange(n - (1 if mode == "eps" else 0) - 6, n - (1 if mode == "eps" else 0), device="cuda")
    if weight == 1.0:                                       # bf16-exact rows: nothing to round
        assert torch.all(ref[exact_rows] == 0) and torch.all(r[exact_rows] == 0)


# ---- 2. eps over every score of every tile --------------------------------------------------------------------------
def _coherent_magnitudes(d, w):
    """``d`` powers of two ``2^f_i`` whose weighted, normalised values ``w 2^f_i / |x|`` sit just below the bf16
    midpoint ``2^f_i (1 + 2^-8)``, so each rounds down by nearly ``u`` of itself: ``sum 4^f_i`` is chosen as
    ``(w / (1 + 2^-8))^2 (1 + 2e-5)``, so ``|x|`` is known exactly and no iteration on the norm is needed.  Most
    entries share one or two exponents; the last 24 make up the remainder."""
    m = 1.0 + 2.0 ** -8
    t0 = (abs(w) / m) ** 2
    target = t0 * (1 + 2e-5)
    nb = d - 24
    f0 = math.floor(math.log(target / nb, 4))
    while nb * 4.0 ** (f0 + 1) <= target:
        f0 += 1
    while nb * 4.0 ** f0 > target:
        f0 -= 1
    n_up = min(nb, int((target - nb * 4.0 ** f0) // (3 * 4.0 ** f0)))
    exps = [f0 + 1] * n_up + [f0] * (nb - n_up)
    rem = target - n_up * 4.0 ** (f0 + 1) - (nb - n_up) * 4.0 ** f0
    for _ in range(d - nb):
        f = math.floor(math.log(rem, 4)) if rem > 4.0 ** (f0 - 20) else f0 - 20
        while 4.0 ** f > rem and f > f0 - 20:
            f -= 1
        exps.append(f)
        rem -= 4.0 ** f
    s = sum(4.0 ** f for f in exps)
    assert 1e-5 < s / t0 - 1 < 3e-5
    return torch.tensor([2.0 ** f for f in exps], dtype=torch.float32, device="cuda")


def _family(name, n_part, n, dims, wts, g):
    """(queries, corpus) raw fp32 rows; corpus rows 0 .. n_part - 1 are the partners of the queries."""
    D = sum(dims)
    if name == "gaussian":
        return torch.randn((n_part, D), generator=g, device="cuda"), torch.randn((n, D), generator=g, device="cuda")
    if name == "coherent":
        # one magnitude pattern per space and side, permuted and signed per row; a query and its partner share
        # permutation and signs, so their rounding errors point the same way and add up in the product
        q = torch.empty((n_part, D), device="cuda")
        v = torch.empty((n, D), device="cuda")
        o = 0
        for d, w in zip(dims, wts):
            mq, mv = _coherent_magnitudes(d, w), _coherent_magnitudes(d, 1.0)
            perm = torch.argsort(torch.rand((n, d), generator=g, device="cuda"), dim=1)
            sign = torch.where(torch.rand((n, d), generator=g, device="cuda") < 0.5, -1.0, 1.0)
            v[:, o:o + d] = mv[perm] * sign
            q[:, o:o + d] = mq[perm[:n_part]] * sign[:n_part]
            o += d
        return q, v
    if name == "cancellation":
        # the partner negates the second half of the query's columns: two partial sums of about +-1/2 per unit weight
        q = torch.randn((n_part, D), generator=g, device="cuda")
        v = torch.randn((n, D), generator=g, device="cuda")
        v[:n_part] = q
        v[:n_part, D // 2:] *= -1
        return q, v
    if name == "heavy":
        # one component of each space carries about 90 % of its norm; the partner shares it
        def heavy(x):
            o = 0
            for d in dims:
                sp = x[:, o:o + d]
                j = torch.randint(0, d, (x.shape[0], 1), generator=g, device="cuda")
                sp.scatter_(1, j, 3.0 * torch.linalg.vector_norm(sp, dim=1, keepdim=True))
                o += d
            return x
        q = heavy(torch.randn((n_part, D), generator=g, device="cuda"))
        v = heavy(torch.randn((n, D), generator=g, device="cuda"))
        v[:n_part] = q + 0.05 * torch.randn((n_part, D), generator=g, device="cuda")
        return q, v
    raise ValueError(name)


# family, dims, weights, norm mode, frames
EPS_CASES = [
    ("gaussian", (1536, 512), (0.6, 0.4), "plain", 1),
    ("gaussian", (6000,), (1.0,), "eps", 1),
    ("gaussian", (1536, 512), (0.6, 0.4), "plain", 4),
    ("coherent", (1536, 512), (0.6, 0.4), "plain", 1),
    ("coherent", (3000, 3000), (1.0, 1.0), "plain", 1),
    ("coherent", (1024, 512, 256), (0.9, 0.05, 0.05), "eps", 1),
    ("coherent", (6000,), (1.0,), "eps", 1),
    ("cancellation", (3000, 3000), (1.0, 1.0), "eps", 1),
    ("cancellation", (6000,), (1.0,), "plain", 1),
    ("cancellation", (1536, 512), (0.6, 0.4), "plain", 2),
    ("heavy", (1024, 512, 256), (0.9, 0.05, 0.05), "plain", 1),
    ("heavy", (1536, 512), (0.6, 0.4), "eps", 1),
]


def _tile_scores(X, a_op, nq, store, kernel, lo_value):
    """fp32 scores [nq, n] of every pair, from ``xmve_score_store`` or from a FILTER window below every score."""
    N, nv = X.N, store.n
    if kernel == "store":
        out = torch.full((nq, nv), float("nan"), dtype=torch.float32, device="cuda")
        N.call("xmve_score_store", N.ptr(a_op), nq, a_op.stride(0), N.ptr(store.op), nv, store.op.stride(0), 1,
               store.k, 1.0, N.ptr(out), nv, N.stream_ptr())
        return out
    cap = nv
    lo = torch.full((nq,), lo_value, dtype=torch.float32, device="cuda")
    cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")
    c_s = torch.zeros((nq, cap), dtype=torch.float32, device="cuda")
    c_i = torch.full((nq, cap), -1, dtype=torch.int32, device="cuda")
    N.call("xmve_score_filter", N.ptr(a_op), nq, a_op.stride(0), N.ptr(store.op), nv, store.op.stride(0), 1, store.k,
           N.ptr(lo), None, None, N.ptr(cnt), N.ptr(c_s), N.ptr(c_i), cap, N.stream_ptr())
    assert torch.all(cnt == nv), "the window lies below every score: every pair is listed"
    idx = c_i.long()
    assert torch.equal(torch.sort(idx, dim=1).values, torch.arange(nv, device="cuda").expand(nq, nv))
    out = torch.full((nq, nv), float("nan"), dtype=torch.float32, device="cuda")
    out.scatter_(1, idx, c_s)
    return out


@pytest.mark.parametrize("family,dims,wts,mode,frames", EPS_CASES,
                         ids=["%s-%s-%s-f%d" % (c[0], "x".join(map(str, c[1])), c[3], c[4]) for c in EPS_CASES])
def test_eps_bounds_every_score_of_every_tile(X, monkeypatch, family, dims, wts, mode, frames):
    E = X.engine
    nq, nv = 200, 8269
    g = _gen(100 + len(dims) * 7 + sum(dims) + frames)
    q, v = _family(family, nq, nv, dims, wts, g)
    if frames > 1:                                          # frame-pooled rows: K1 averages T frames per row
        q = q.unsqueeze(1) + 0.5 * torch.randn((nq, frames, q.shape[1]), generator=g, device="cuda")
        v = v.unsqueeze(1) + 0.5 * torch.randn((nv, frames, v.shape[1]), generator=g, device="cuda")
    store = E.CorpusStore(nv, dims, norm_mode=mode).add(v)
    a_op, _, _, q_res, _ = store.prepare_queries(q, wts)
    eps = float(E._eps_device(q_res, E._dv2_global([store], E.SoloComm()), wts, len(dims), store.k))
    w_norm = math.sqrt(sum(w * w for w in wts))
    if family == "coherent":                                # the construction worked: queries round by about u
        dq = q_res[:, :nq].double().sum(0).sqrt()
        assert float(dq.min()) >= 0.8 * U * w_norm, float(dq.min()) / (U * w_norm)
    exact = _exact(_pool(q), _pool(v), dims, wts, mode)
    qb, vb = a_op[:nq].double(), store.op[:nv].double()
    dot = qb @ vb.T                                         # <Qb, Vb> in fp64: exact products, negligible sum error
    acc = store.k * 2.0 ** -22 * torch.linalg.vector_norm(qb, dim=1)[:, None] * torch.linalg.vector_norm(vb, dim=1)
    lo_value = -(sum(abs(w) for w in wts) + 1.0)
    for tile in TILES:
        monkeypatch.setenv("XMVE_TILE", str(tile))
        for kernel in ("store", "filter"):
            s = _tile_scores(X, a_op, nq, store, kernel, lo_value).double()
            torch.cuda.synchronize()
            assert not torch.isnan(s).any()
            err = (s - exact).abs()
            err_acc = (s - dot).abs()
            r_eps, r_acc = float(err.max()) / eps, float((err_acc / acc).max())
            print("eps-bound %-12s %-14s %-5s norm=%s frames=%d tile=%d %-6s eps=%.4e max err/eps=%.4f "
                  "max err/acc-term=%.4f" % (family, "x".join(map(str, dims)), ",".join(map(str, wts)), mode,
                                             frames, tile, kernel, eps, r_eps, r_acc))
            assert r_eps <= 1.0, "tile %d %s: |approx - exact| reaches %.4g eps" % (tile, kernel, r_eps)
            assert r_acc <= 1.0, "tile %d %s: fp32 accumulation error reaches %.4g of K 2^-22 |Qb||Vb|" % (
                tile, kernel, r_acc)


# ---- 3. exact answers inside eps ----------------------------------------------------------------------------------
L = 0.6
CLUSTER = 2000


def _cluster_corpus(q, dims, wts, half_width, n_fill, g):
    """Per query ``j``, rows ``j*CLUSTER ..`` whose fused scores spread evenly over ``[L - hw, L + hw]``: per space
    ``c q_hat + sqrt(1 - c^2) r`` with ``r`` a unit vector orthogonal to ``q_hat`` (the weights sum to 1, so the fused
    score is ``c``); then ``n_fill`` Gaussian rows, whose scores lie far below ``L``."""
    nq, D = q.shape
    c = torch.linspace(L - half_width, L + half_width, CLUSTER, dtype=torch.float64, device="cuda")
    c = c[torch.randperm(CLUSTER, generator=g, device="cuda")]
    parts = []
    for j in range(nq):
        rows, o = [], 0
        for d in dims:
            qh = _unit(q[j:j + 1, o:o + d].double(), "plain")
            r = torch.randn((CLUSTER, d), generator=g, device="cuda", dtype=torch.float64)
            r = _unit(r - (r @ qh.T) * qh, "plain")
            rows.append(c[:, None] * qh + (1 - c * c).sqrt()[:, None] * r)
            o += d
        parts.append(torch.cat(rows, 1).float())
    parts.append(torch.randn((n_fill, D), generator=g, device="cuda"))
    return torch.cat(parts)


def _order(s):
    """Row indices by (score desc, row asc); NaN last."""
    s = torch.nan_to_num(s, nan=-math.inf)
    return torch.argsort(-s, dim=1, stable=True)


def _inversions(approx, exact):
    """Fraction of pairs of a cluster that the fp32 scores order differently from the fp64 scores."""
    o = torch.argsort(exact)
    a = approx[o]
    n = a.numel()
    inv = (a[:, None] > a[None, :]).triu(1).sum()
    return float(inv) / (n * (n - 1) / 2)


def _check_topk(s, i, exact, k, eligible=None):
    ex = exact.clone()
    if eligible is not None:
        ex[~eligible] = -math.inf
    ref = _order(ex)[:, :k]
    assert torch.equal(i, ref), "top-k differs from the fp64 oracle in %d of %d rows" % (
        int((i != ref).any(1).sum()), i.shape[0])
    assert float((s - torch.gather(ex, 1, ref)).abs().max()) <= 1e-13


@pytest.fixture(scope="module", params=["plain", "eps"])
def cluster(X, request):
    E, mode = X.engine, request.param
    dims, wts = (1536, 512), (0.6, 0.4)
    nq, n_fill = 8, 24000
    g = _gen(501 if mode == "plain" else 502)
    q = torch.randn((nq, sum(dims)), generator=g, device="cuda")
    pre = E.CorpusStore(4096, dims, norm_mode=mode).add(torch.randn((4096, sum(dims)), generator=g, device="cuda"))
    _, _, _, q_res, _ = pre.prepare_queries(q, wts)
    eps0 = float(E._eps_device(q_res, E._dv2_global([pre], E.SoloComm()), wts, 2, pre.k))
    v = _cluster_corpus(q, dims, wts, eps0 / 8, n_fill, g)
    store = E.CorpusStore(len(v), dims, norm_mode=mode).add(v)
    exact = _exact(q, v, dims, wts, mode)
    return dict(E=E, dims=dims, wts=wts, mode=mode, q=q, v=v, store=store, exact=exact, eps0=eps0, nq=nq)


def test_cluster_is_adversarial(X, cluster):
    """At least 5 % of each cluster's pairs are ordered differently by the fp32 tensor-core scores."""
    c, E = cluster, cluster["E"]
    store = c["store"]
    a_op, _, _, q_res, nq = store.prepare_queries(c["q"], c["wts"])
    eps = float(E._eps_device(q_res, E._dv2_global([store], E.SoloComm()), c["wts"], 2, store.k))
    approx = _tile_scores(X, a_op, nq, store, "store", 0.0).double()
    fracs = []
    for j in range(nq):
        sl = slice(j * CLUSTER, (j + 1) * CLUSTER)
        ex = c["exact"][j, sl]
        assert float(ex.max() - ex.min()) <= c["eps0"] / 4 + 1e-6    # the cluster lies within +-eps/8 of L
        fracs.append(_inversions(approx[j, sl], ex))
    print("cluster %s: eps %.4e, inversion fraction per query %s" % (c["mode"], eps,
                                                                     " ".join("%.3f" % f for f in fracs)))
    assert min(fracs) >= 0.05


@pytest.mark.parametrize("small_nv", [0, None])
def test_search_inside_eps(cluster, small_nv):
    c = cluster
    kw = {} if small_nv is None else {"small_nv": small_nv}
    for k in (1, 700, 1000, 1999):
        s, i = c["store"].search(c["q"], k, weights=c["wts"], **kw)
        _check_topk(s, i, c["exact"], k)


def test_search_shards_inside_eps(cluster):
    c, E = cluster, cluster["E"]
    v, n = c["v"], c["v"].shape[0]
    cuts = [0, n // 3 + 5, 2 * n // 3 - 7, n]
    shards = [E.CorpusStore(b - a, c["dims"], norm_mode=c["mode"], index_offset=a).add(v[a:b])
              for a, b in zip(cuts[:-1], cuts[1:])]
    s, i = E.search_shards(shards, c["q"], 1000, weights=c["wts"])
    _check_topk(s, i, c["exact"], 1000)


def test_filtered_and_excluded_search_inside_eps(cluster):
    c, E = cluster, cluster["E"]
    n = c["v"].shape[0]
    labels = torch.arange(n, device="cuda") % 2                        # half of every cluster is ineligible
    store = E.CorpusStore(n, c["dims"], norm_mode=c["mode"]).add(c["v"], labels=labels)
    s, i = store.search(c["q"], 600, weights=c["wts"], label_mask=1)
    _check_topk(s, i, c["exact"], 600, eligible=(labels == 0)[None, :].expand(c["nq"], n))
    ref = _order(c["exact"])
    excl = ref[:, 500]                      # a cluster row inside the list; a strided view, as callers pass them
    s, i = c["store"].search(c["q"], 800, weights=c["wts"], exclude=excl)
    elig = torch.ones_like(c["exact"], dtype=torch.bool)
    elig[torch.arange(c["nq"], device="cuda"), excl] = False
    _check_topk(s, i, c["exact"], 800, eligible=elig)


def test_graph_search_inside_eps(cluster):
    c, E = cluster, cluster["E"]
    gs = E.GraphSearch(c["store"], c["nq"], 1000, weights=c["wts"])
    for _ in range(2):
        s, i = gs(c["q"])
        _check_topk(s, i, c["exact"], 1000)


def test_range_search_and_count_inside_eps(cluster):
    c = cluster
    ex = c["exact"]
    top = torch.sort(ex, dim=1, descending=True).values
    pos = torch.tensor([250, 999, 1000, 1777, 1, 1500, 640, 1999][:c["nq"]], device="cuda")
    ms = 0.5 * (top.gather(1, pos[:, None] - 1) + top.gather(1, pos[:, None])).flatten()
    res = c["store"].range_search(c["q"], ms.cpu().numpy(), weights=c["wts"])
    cnt = c["store"].range_count(c["q"], ms.cpu().numpy(), weights=c["wts"])
    off = res.offsets
    assert torch.equal(cnt, off[1:] - off[:-1])
    ref = _order(ex)
    for j in range(c["nq"]):
        n = int(pos[j])
        assert int(cnt[j]) == n
        assert torch.equal(res.idx[off[j]:off[j + 1]], ref[j, :n])
        assert float((res.scores[off[j]:off[j + 1]] - ex[j, ref[j, :n]]).abs().max()) <= 1e-13
    excl = ref[:, 3]                                        # a strided view: one row per query, inside most lists
    res = c["store"].range_search(c["q"], ms.cpu().numpy(), weights=c["wts"], exclude=excl)
    cnt = c["store"].range_count(c["q"], ms.cpu().numpy(), weights=c["wts"], exclude=excl)
    off = res.offsets
    assert torch.equal(cnt, off[1:] - off[:-1])
    for j in range(c["nq"]):
        want = ref[j, :int(pos[j])]
        want = want[want != excl[j]]
        assert torch.equal(res.idx[off[j]:off[j + 1]], want), "query %d" % j


def test_rank_of_gt_inside_eps(cluster):
    c, E = cluster, cluster["E"]
    ex = c["exact"]
    g = torch.Generator().manual_seed(9)
    off, rows = [0], []
    for j in range(c["nq"]):
        picks = (j * CLUSTER + torch.randperm(CLUSTER, generator=g)[:6]).tolist() + [c["v"].shape[0] - 1 - j]
        rows += picks
        off.append(len(rows))
    ranks = E.rank_of_gt([c["store"]], c["q"], off, rows, weights=c["wts"])
    # the position in the stable ascending argsort of the fp64 errors (the negated scores)
    pos = torch.empty_like(ex, dtype=torch.int64)
    o = torch.argsort(-ex, dim=1, stable=True)
    pos.scatter_(1, o, torch.arange(ex.shape[1], device="cuda").expand_as(o))
    want = [int(pos[j, r]) + 1 for j in range(c["nq"]) for r in rows[off[j]:off[j + 1]]]
    assert ranks.cpu().tolist() == want


def test_similar_pairs_inside_eps(X, cluster):
    """A band of near-duplicate rows whose pair scores spread over about eps / 2 around ``min_score``."""
    c, E = cluster, cluster["E"]
    dims, wts, mode = c["dims"], c["wts"], c["mode"]
    g = _gen(77)
    D, nb, n_fill = sum(dims), 500, 16000
    p = torch.randn((1, D), generator=g, device="cuda", dtype=torch.float64)
    t2 = 0.05 + c["eps0"] * (torch.rand((nb, 1), generator=g, device="cuda", dtype=torch.float64) - 0.5) / 2
    rows, o = [], 0
    for d in dims:                                          # cos(v_i, v_j) ~ 1 - (t_i^2 + t_j^2) / 2 per space
        ph = _unit(p[:, o:o + d], "plain")
        r = torch.randn((nb, d), generator=g, device="cuda", dtype=torch.float64)
        r = _unit(r - (r @ ph.T) * ph, "plain")
        rows.append(ph + t2.sqrt() * r)
        o += d
    v = torch.cat([torch.cat(rows, 1).float(), torch.randn((n_fill, D), generator=g, device="cuda")])
    v = v[torch.randperm(len(v), generator=g, device="cuda")]
    ex = _exact(v, v, dims, wts, mode)
    up = ex.triu(1)
    vals = torch.sort(up[up > 0.5], descending=True).values
    jj = vals.numel() // 2
    ms = float(0.5 * (vals[jj - 1] + vals[jj]))
    assert int(((vals - ms).abs() < c["eps0"]).sum()) >= 2000              # thousands of pairs within eps of it
    store = E.CorpusStore(len(v), dims, norm_mode=mode).add(v)
    res = store.similar_pairs(ms, weights=wts)
    off = res.offsets
    total = 0
    for i in range(len(v)):
        want = (ex[i] >= ms) & (torch.arange(len(v), device="cuda") > i)
        n = int(want.sum())
        got = res.idx[off[i]:off[i + 1]]
        assert got.numel() == n, "row %d" % i
        if n:
            o = _order(torch.where(want, ex[i], torch.full_like(ex[i], -math.inf))[None])[0, :n]
            assert torch.equal(got, o)
            assert float((res.scores[off[i]:off[i + 1]] - ex[i, o]).abs().max()) <= 1e-13
        total += n
    assert total == jj


def test_zero_row_takes_the_a_priori_bound(X):
    """A zero row under 'plain' makes its residual NaN: eps becomes the a-priori bound (d = 4096 is past the K where a
    constant 8.5e-3 fell below it).  Searches stay exact inside that eps and never return the zero row."""
    E = X.engine
    d, nq = 4096, 6
    g = _gen(901)
    q = torch.randn((nq, d), generator=g, device="cuda")
    hw = E.eps_fallback((1.0,), 1, d) / 8
    v = _cluster_corpus(q, (d,), (1.0,), hw, 12000, g)
    zero = 4321
    v[zero] = 0
    store = E.CorpusStore(len(v), (d,)).add(v)
    _, _, _, q_res, _ = store.prepare_queries(q, (1.0,))
    eps = float(E._eps_device(q_res, E._dv2_global([store], E.SoloComm()), (1.0,), 1, store.k))
    assert eps == E.eps_fallback((1.0,), 1, store.k)
    exact = _exact(q, v, (d,), (1.0,), "plain")
    assert torch.isnan(exact[:, zero]).all()
    for kw in ({}, {"small_nv": 0}):
        for k in (1000, 1999):
            s, i = store.search(q, k, **kw)
            assert not (i == zero).any()
            _check_topk(s, i, exact, k)
