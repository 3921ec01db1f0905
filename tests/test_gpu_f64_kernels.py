"""The fp64 evaluation kernels (B200 only): score matrix, pairwise measures, triplet cost, ground-truth ranks,
norm_score and the band counts of the rank-of-ground-truth path, each called through the C ABI and compared with a
plain NumPy statement of the same operation, at the tile edges, strides and values where tiled kernels go wrong.

Floating-point results are held to a bound derived from the operation, not to a fixed tolerance: a dot product of
length k summed in any order by fused multiply-adds is within gamma_k * sum_i |a_i b_i| of the exact value,
gamma_k = k u / (1 - k u), u = 2^-53.  Integer results (ranks, counts) and the element-wise epilogues must be exact.
Operands and outputs sit inside larger buffers whose unused rows and columns hold values that would change the result
if a kernel read them (NaN, -inf, +inf) or that it must leave alone (a sentinel)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
SENTINEL = -12345.5


@pytest.fixture(scope="module")
def N():
    from cross_modal_video_engine_b200 import _native
    _native.require_device()
    return _native


def _gamma(k):
    return k * U / (1 - k * U)


def _buffer(vals, ld, fill, extra_rows=1):
    """Device copy of the 2-D array ``vals`` as the top-left corner of a [rows + extra_rows, ld] buffer of ``fill``."""
    rows, cols = vals.shape
    buf = np.full((rows + extra_rows, ld), fill, dtype=vals.dtype)
    buf[:rows, :cols] = vals
    return torch.from_numpy(buf).cuda()


# The three fp64 score kernels; XMVE_F64_KERNEL and XMVE_F64_BK are read on every call.  Odd operand strides route
# every variant to the FMA kernel.
F64_VARIANTS = {"fma": {"XMVE_F64_KERNEL": "fma"}, "dmma32": {}, "dmma16": {"XMVE_F64_BK": "16"}}


def _use_variant(monkeypatch, name):
    monkeypatch.delenv("XMVE_F64_KERNEL", raising=False)
    monkeypatch.delenv("XMVE_F64_BK", raising=False)
    for key, val in F64_VARIANTS[name].items():
        monkeypatch.setenv(key, val)


def _score_f64(N, a, nq, a_ld, b, nv, b_ld, k, alpha, out_ld):
    out = torch.full((nq + 1, out_ld), SENTINEL, dtype=torch.float64, device="cuda")
    N.call("xmve_score_f64", N.ptr(a), nq, a_ld, N.ptr(b), nv, b_ld, k, alpha, N.ptr(out), out_ld, N.stream_ptr())
    return out.cpu().numpy()


# ---- xmve_score_f64 ------------------------------------------------------------------------------------------------
# (nq, nv, k, a_ld - k, b_ld - k, out_ld - nv, alpha).  nq and nv run over 1, 63, 64, 65, 127, 128, 129 and 300 (the
# 128 x 64 block tile), k over 1, 2, 3, 4, 31, 32, 33, 200 and 1537 (the k-blocks of 16 and 32; an odd k makes the
# DMMA producer copy 8 bytes and zero-fill the other 8).  An odd stride sends all three variants to the FMA kernel.
SCORE_CASES = [
    (1, 300, 1, 1, 1, 2, -1.0),
    (300, 1, 1, 0, 0, 0, -1.0),
    (63, 64, 2, 0, 0, 1, -1.0),
    (64, 65, 3, 1, 1, 3, -1.0),
    (65, 63, 4, 0, 2, 0, 0.3),
    (127, 129, 31, 1, 1, 1, -1.0),
    (128, 128, 32, 0, 0, 2, -1.0),
    (129, 127, 33, 3, 1, 0, -1.0),
    (129, 65, 33, 0, 0, 1, -1.0),
    (300, 300, 200, 2, 4, 3, -1.0),
    (64, 63, 200, 1, 0, 0, -1.0),
    (65, 129, 1537, 1, 1, 1, -1.0),
    (127, 128, 1537, 0, 0, 2, 0.3),
    (1, 1, 31, 0, 0, 0, -1.0),
]


@pytest.mark.parametrize("nq,nv,k,a_pad,b_pad,out_pad,alpha", SCORE_CASES)
def test_score_f64_within_the_dot_product_bound(N, monkeypatch, nq, nv, k, a_pad, b_pad, out_pad, alpha):
    rng = np.random.default_rng(nq * 7919 + nv * 31 + k)
    A, B = rng.standard_normal((nq, k)), rng.standard_normal((nv, k))
    a_ld, b_ld, out_ld = k + a_pad, k + b_pad, nv + out_pad
    a, b = _buffer(A, a_ld, np.nan), _buffer(B, b_ld, np.nan)
    ref = (A.astype(np.longdouble) @ B.astype(np.longdouble).T) * alpha
    mag = np.abs(A) @ np.abs(B).T * (1 + 1e-9)
    bound = abs(alpha) * (_gamma(k) + 2.0 ** -60) * mag + U * np.abs(ref).astype(np.float64) + 1e-300
    for variant in F64_VARIANTS:
        _use_variant(monkeypatch, variant)
        out = _score_f64(N, a, nq, a_ld, b, nv, b_ld, k, alpha, out_ld)
        err = np.abs((out[:nq, :nv].astype(np.longdouble) - ref).astype(np.float64))
        assert np.all(err <= bound), (variant, float((err / bound).max()))
        assert np.all(out[:nq, nv:] == SENTINEL) and np.all(out[nq] == SENTINEL), variant   # padding untouched


# ---- xmve_score_f64_fused -----------------------------------------------------------------------------------------
# (nq, nv, k, out_ld, out_off): even out_ld on an aligned output takes the 16-byte store, odd out_ld or an output one
# double off alignment the scalar store, and with an odd nv the last column is scalar in either case.
FUSED_CASES = [(129, 65, 33, 66, 0), (64, 63, 200, 63, 0), (127, 128, 32, 130, 1), (300, 129, 64, 130, 0),
               (65, 1, 3, 1, 0)]


@pytest.mark.parametrize("variant", ["dmma32", "dmma16"])
@pytest.mark.parametrize("nq,nv,k,out_ld,out_off", FUSED_CASES)
def test_score_f64_fused_is_the_numpy_fusion_of_the_stored_matrix(N, monkeypatch, variant, nq, nv, k, out_ld, out_off):
    """first = 1: w * e, first = 0: acc + w * e, bit for bit, with e the matrix xmve_score_f64 stores (same kernel)."""
    _use_variant(monkeypatch, variant)
    rng = np.random.default_rng(nq + nv + k)
    A, B = rng.standard_normal((nq, k)), rng.standard_normal((nv, k))
    a_ld = b_ld = k + (k % 2)
    a, b = _buffer(A, a_ld, np.nan), _buffer(B, b_ld, np.nan)
    alpha, w = -1.0, 0.37
    e = _score_f64(N, a, nq, a_ld, b, nv, b_ld, k, alpha, nv)[:nq, :nv]
    acc0 = rng.standard_normal((nq, nv))
    for first in (1, 0):
        flat = np.full(out_off + (nq + 1) * out_ld, SENTINEL)
        flat[out_off:out_off + nq * out_ld].reshape(nq, out_ld)[:, :nv] = acc0
        buf = torch.from_numpy(flat).cuda()
        out = buf[out_off:]
        N.call("xmve_score_f64_fused", N.ptr(a), nq, a_ld, N.ptr(b), nv, b_ld, k, alpha, w, first, N.ptr(out), out_ld,
               N.stream_ptr())
        got = buf.cpu().numpy()
        mat = got[out_off:out_off + nq * out_ld].reshape(nq, out_ld)
        want = w * e if first else acc0 + w * e
        assert np.array_equal(mat[:, :nv], want), (first, int((mat[:, :nv] != want).sum()))
        assert np.all(mat[:, nv:] == SENTINEL) and np.all(got[:out_off] == SENTINEL)
        assert np.all(got[out_off + nq * out_ld:] == SENTINEL)


def test_score_f64_fused_refuses_unaligned_operands(N, monkeypatch):
    _use_variant(monkeypatch, "dmma32")
    nq, nv, k = 20, 30, 33
    a = torch.randn((nq + 1, k + 1), dtype=torch.float64, device="cuda")
    b = torch.randn((nv + 1, k + 1), dtype=torch.float64, device="cuda")
    out = torch.zeros((nq, nv), dtype=torch.float64, device="cuda")
    args = (k, -1.0, 0.5, 1, N.ptr(out), nv, N.stream_ptr())
    st = N.lib.xmve_score_f64_fused(N.ptr(a), nq, k, N.ptr(b), nv, k + 1, *args)             # odd a_ld
    assert st == -1                                                                          # XMVE_ERR_ARG
    st = N.lib.xmve_score_f64_fused(N.ptr(a), nq, k + 1, N.ptr(b), nv, k, *args)             # odd b_ld
    assert st == -1
    a1 = a.view(-1)[1:]                                                                      # 8 bytes off alignment
    st = N.lib.xmve_score_f64_fused(N.ptr(a1), nq, k + 1, N.ptr(b), nv, k + 1, *args)
    assert st == -1
    torch.cuda.synchronize()
    assert bool((out == 0).all())                                                            # nothing was launched


# ---- xmve_pairwise_f64 --------------------------------------------------------------------------------------------
MEASURES = ["L1", "L2", "JACCARD", "SQL2", "DOT", "ORDER"]


def _pairwise_reference(measure, A, B):
    """(f, error bound of the kernel's f) in long double; f as the header comment of xmve_pairwise_f64 states it."""
    a = A.astype(np.longdouble)[:, None, :]
    b = B.astype(np.longdouble)[None, :, :]
    k = A.shape[1]
    if measure == "JACCARD":
        p, q = np.minimum(a, b).sum(-1), np.maximum(a, b).sum(-1)
        f = p / q
        return f, (_gamma(k) * (p + f * q) / (q * (1 - _gamma(k))) + U * f).astype(np.float64)
    if measure == "DOT":
        t = a * b
        return t.sum(-1), (_gamma(k) * np.abs(t).sum(-1)).astype(np.float64)
    if measure == "L1":
        t = np.abs(a - b)                          # the kernel rounds each difference, then sums
        return t.sum(-1), (_gamma(k + 1) * t.sum(-1)).astype(np.float64)
    t = np.maximum(b - a, 0) ** 2 if measure == "ORDER" else (a - b) ** 2
    s = t.sum(-1)
    es = _gamma(k + 2) * s                          # a rounded difference squared: two more roundings per term
    if measure == "SQL2":
        return s, es.astype(np.float64)
    f = np.sqrt(s)                                  # |sqrt(s') - sqrt(s)| = |s' - s| / (sqrt(s') + sqrt(s))
    den = f + np.sqrt(np.maximum(s - es, 0))
    ef = np.where(den > 0, es / np.where(den > 0, den, 1), np.sqrt(es))
    return f, (ef + U * f).astype(np.float64)


# (nq, nv, k, a_ld - k, b_ld - k) around the 64 x 64 x 16 tile
PAIR_CASES = [(1, 1, 1, 0, 0), (63, 65, 15, 1, 0), (64, 64, 16, 0, 3), (65, 63, 17, 2, 1), (129, 64, 33, 0, 0),
              (64, 129, 200, 5, 0), (3, 130, 64, 0, 0)]


@pytest.mark.parametrize("measure", MEASURES)
@pytest.mark.parametrize("nq,nv,k,a_pad,b_pad", PAIR_CASES)
def test_pairwise_f64_within_the_bound_of_its_sum(N, measure, nq, nv, k, a_pad, b_pad):
    rng = np.random.default_rng(nq * 1000 + nv + k)
    A, B = rng.standard_normal((nq, k)), rng.standard_normal((nv, k))
    if measure == "JACCARD":                                  # loss.jaccard_sim is meant for non-negative features
        A, B = np.abs(A) + 0.01, np.abs(B) + 0.01
    n_same = min(nq, nv, 3)
    B[:n_same] = A[:n_same]                                   # identical rows: distance exactly 0
    a_ld, b_ld = k + a_pad, k + b_pad
    a, b = _buffer(A, a_ld, np.nan), _buffer(B, b_ld, np.nan)
    f, ef = _pairwise_reference(measure, A, B)
    forms = [(1.0, 0.0)]
    if measure in ("L1", "L2"):
        forms.append((-1.0 / k, -1.0))                        # 'l1_norm' / 'l2_norm' of cal_error
    if measure == "JACCARD":
        forms.append((-1.0, 0.0))
    code = getattr(N, "MEASURE_" + measure)
    for alpha, beta in forms:
        out = torch.full((nq + 1, nv + 2), SENTINEL, dtype=torch.float64, device="cuda")
        N.call("xmve_pairwise_f64", N.ptr(a), nq, a_ld, N.ptr(b), nv, b_ld, k, code, alpha, beta, N.ptr(out), nv + 2,
               N.stream_ptr())
        got = out.cpu().numpy()
        ref = f * alpha + beta
        bound = abs(alpha) * ef * (1 + 4 * U) + 2 * U * (np.abs(alpha * f).astype(np.float64) + abs(beta)) + 1e-300
        err = np.abs((got[:nq, :nv].astype(np.longdouble) - ref).astype(np.float64))
        assert np.all(err <= bound), (alpha, beta, float((err / bound).max()))
        assert np.all(got[:nq, nv:] == SENTINEL) and np.all(got[nq] == SENTINEL)
        if measure in ("L1", "L2", "SQL2") and alpha == 1.0:
            assert np.all(np.diagonal(got[:n_same, :n_same]) == 0.0)


@pytest.mark.parametrize("measure", ["L1", "L2", "SQL2", "DOT"])
def test_pairwise_f64_nan_stays_in_its_row_and_column(N, measure):
    rng = np.random.default_rng(3)
    nq, nv, k = 70, 130, 33
    A, B = rng.standard_normal((nq, k)), rng.standard_normal((nv, k))
    A[5, 32] = np.nan                                         # in the last, partial k-block
    B[64, 0] = np.nan                                         # first row of the second column tile
    a, b = _buffer(A, k + 1, 0.0), _buffer(B, k, 0.0)
    out = torch.empty((nq, nv), dtype=torch.float64, device="cuda")
    N.call("xmve_pairwise_f64", N.ptr(a), nq, k + 1, N.ptr(b), nv, k, k, getattr(N, "MEASURE_" + measure), 1.0, 0.0,
           N.ptr(out), nv, N.stream_ptr())
    nan = np.isnan(out.cpu().numpy())
    want = np.zeros((nq, nv), bool)
    want[5, :] = True
    want[:, 64] = True
    assert np.array_equal(nan, want)


# ---- xmve_triplet_cost --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2, 255, 256, 257])
@pytest.mark.parametrize("margin", [0.0, 0.2])
@pytest.mark.parametrize("max_violation", [0, 1])
def test_triplet_cost_matches_numpy(N, n, margin, max_violation):
    rng = np.random.default_rng(n)
    S = rng.uniform(-1.0, 1.0, (n, n))
    S[np.arange(n), np.arange(n)] = rng.uniform(0.0, 1.0, n)
    scores = _buffer(S, n + 3, np.nan)                        # ld > n; the padding would poison a sum
    d = np.diagonal(S)
    cost_s = np.maximum(margin + S - d[:, None], 0.0)
    cost_im = np.maximum(margin + S - d[None, :], 0.0)
    np.fill_diagonal(cost_s, 0.0)
    np.fill_diagonal(cost_im, 0.0)
    if max_violation:
        want = [cost_s.max(1).sum(), cost_im.max(0).sum()]
    else:
        want = [cost_s.sum(), cost_im.sum()]
    out = torch.full((2,), np.nan, dtype=torch.float64, device="cuda")
    N.call("xmve_triplet_cost", N.ptr(scores), n, n + 3, margin, max_violation, N.ptr(out), N.stream_ptr())
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-12, atol=0)


# ---- xmve_gt_ranks ------------------------------------------------------------------------------------------------
def _stable_ranks(line, ids):
    """1-based position of each id in np.argsort(line, kind="stable"): NaN after every number, -0.0 == +0.0."""
    pos = np.empty(line.size, np.int64)
    pos[np.argsort(line, kind="stable")] = np.arange(line.size)
    return pos[ids] + 1


def _rank_problem(dtype, axis, max_gt, seed):
    """Tie-heavy errors (8 levels, +-0.0, +-inf, NaN), a whole-NaN query line and a CSR with empty queries, duplicate
    ids and NaN ground truths.  axis 0: 200 queries x 1000 memories; axis 1: 4000 memories x 40 queries, which the
    column kernel splits into many row slices."""
    rng = np.random.default_rng(seed)
    n_row, n_col = (200, 1000) if axis == 0 else (4000, 40)
    x = ((rng.integers(0, 8, (n_row, n_col)) - 4) * 0.5).astype(dtype)
    u = rng.random((n_row, n_col))
    x[(u < 0.5) & (x == 0)] = -0.0
    x[u > 0.98] = np.inf
    x[(u > 0.96) & (u <= 0.98)] = -np.inf
    x[(u > 0.93) & (u <= 0.96)] = np.nan
    lines = x if axis == 0 else x.T                           # lines[q] = query q's errors
    n_query, n_mem = lines.shape
    lines[3] = np.nan                                         # a zero embedding normalised without epsilon
    sizes = rng.integers(0, max_gt + 1, n_query)
    sizes[[0, 7]] = 0
    sizes[1] = max_gt
    sizes[3] = max(sizes[3], 1)
    ids = []
    for q in range(n_query):
        row = rng.integers(0, n_mem, sizes[q])
        if sizes[q] >= 2:
            row[1] = row[0]                                   # the same id twice
        nan_pos = np.flatnonzero(np.isnan(lines[q]))
        if sizes[q] >= 3 and nan_pos.size:
            row[2] = rng.choice(nan_pos)                      # a NaN ground truth
        ids.append(row)
    off = np.zeros(n_query + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    return x, lines, off, np.concatenate(ids).astype(np.int32)


def _gt_ranks(N, x, axis, off, ids, max_gt):
    n_row, n_col = x.shape
    xd = _buffer(x, n_col + 5, -np.inf)                       # ld > n_col; an extra row and padding of -inf
    off_d, ids_d = torch.from_numpy(off).cuda(), torch.from_numpy(ids).cuda()
    ranks = torch.full((ids.size,), -7, dtype=torch.int32, device="cuda")
    N.call("xmve_gt_ranks", N.ptr(xd), N.F64 if x.dtype == np.float64 else N.F32, n_row, n_col, n_col + 5, axis,
           N.ptr(off_d), N.ptr(ids_d), off.size - 1, ids.size, max_gt, N.ptr(ranks), N.stream_ptr())
    return ranks, off_d


@pytest.mark.parametrize("max_gt", [1, 8, 9, 31, 32, 63, 100])
@pytest.mark.parametrize("axis", [0, 1])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gt_ranks_are_numpy_stable_argsort_positions(N, dtype, axis, max_gt):
    x, lines, off, ids = _rank_problem(dtype, axis, max_gt, seed=max_gt * 4 + axis)
    ranks, _ = _gt_ranks(N, x, axis, off, ids, max_gt)
    want = np.concatenate([_stable_ranks(lines[q], ids[off[q]:off[q + 1]]) for q in range(off.size - 1)])
    got = ranks.cpu().numpy()
    is_nan = np.concatenate([np.isnan(lines[q][ids[off[q]:off[q + 1]]]) for q in range(off.size - 1)])
    bad = np.flatnonzero(got != want)
    assert not np.any(~is_nan[bad]), ("numeric ground truths", bad[~is_nan[bad]][:10])
    assert bad.size == 0, ("NaN ground truths", bad[:10])


@pytest.mark.parametrize("axis", [0, 1])
def test_gt_ranks_of_nan_ground_truths(N, axis):
    """A NaN ground truth (the row of a zero embedding after l2norm) is ranked behind every number, as NumPy's
    argsort ranks it; the whole-NaN query's entries rank in index order among the NaNs."""
    x, lines, off, ids = _rank_problem(np.float64, axis, 9, seed=77)
    ranks, _ = _gt_ranks(N, x, axis, off, ids, 9)
    got = ranks.cpu().numpy()
    q = 3
    g = ids[off[q]:off[q + 1]]
    assert np.array_equal(got[off[q]:off[q + 1]], g + 1)
    is_nan = np.concatenate([np.isnan(lines[p][ids[off[p]:off[p + 1]]]) for p in range(off.size - 1)])
    assert is_nan.sum() > 20
    want = np.concatenate([_stable_ranks(lines[p], ids[off[p]:off[p + 1]]) for p in range(off.size - 1)])
    assert np.array_equal(got[is_nan], want[is_nan])


def test_rank_metrics_on_tie_heavy_ranks(N):
    from cross_modal_video_engine_b200 import metrics
    from test_gpu_kernels import _ap_reference
    max_gt = 9
    x, lines, off, ids = _rank_problem(np.float64, 0, max_gt, seed=5)
    ranks, off_d = _gt_ranks(N, x, 0, off, ids, max_gt)
    n_query, n_mem = lines.shape
    lists = [_stable_ranks(lines[q], ids[off[q]:off[q + 1]]).tolist() for q in range(n_query)]
    for first_only, ap_k in ((False, 0), (False, 10), (True, 0)):
        best = torch.empty(n_query, dtype=torch.int32, device="cuda")
        ap = torch.empty(n_query, dtype=torch.float64, device="cuda")
        tallies = torch.zeros(4, dtype=torch.int64, device="cuda")
        hist = torch.zeros(n_mem + 2, dtype=torch.int32, device="cuda")
        metrics.rank_metrics(ranks, off_d, n_query, n_mem, first_only, ap_k, max_gt, best, ap, tallies, hist)
        want_best = [min(l) if l else n_mem + 1 for l in lists]
        assert best.cpu().tolist() == want_best
        assert ap.cpu().tolist() == [_ap_reference(l, n_mem, ap_k, first_only) for l in lists]
        assert tallies.cpu().tolist() == [sum(b <= t for b in want_best) for t in (1, 5, 10)] + [sum(want_best)]
        assert np.array_equal(hist.cpu().numpy(), np.bincount(want_best, minlength=n_mem + 2))


# ---- xmve_norm_score ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["random", "constant", "nan", "+inf", "-inf", "+-inf"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_norm_score_matches_the_oracle(N, dtype, case):
    """validate.py:7-11 on the same array, NaN and inf included: a NaN anywhere makes every output NaN (np.min /
    np.max propagate it), an error of +inf makes min(-E) = -inf and so max(-E - min) = NaN."""
    from oracle import linas
    rng = np.random.default_rng(11)
    n_row, n_col, ld, out_ld = 300, 1100, 1103, 1101          # more elements than the grid has threads
    E = rng.uniform(-1.0, 1.0, (n_row, n_col)).astype(dtype)
    if case == "constant":
        E[:] = dtype(0.25)
    elif case == "nan":
        E[17, 400] = np.nan
    elif case in ("+inf", "+-inf"):
        E[250, 3] = np.inf
    if case in ("-inf", "+-inf"):
        E[0, 1099] = -np.inf
    x = _buffer(E, ld, np.nan)
    out = torch.full((n_row + 1, out_ld), SENTINEL, dtype=x.dtype, device="cuda")
    scratch = torch.empty(2, dtype=torch.float64, device="cuda")
    N.call("xmve_norm_score", N.ptr(x), N.F64 if dtype == np.float64 else N.F32, n_row, n_col, ld, N.ptr(out), out_ld,
           N.ptr(scratch), N.stream_ptr())
    got = out.cpu().numpy()
    with np.errstate(all="ignore"):
        want = linas.norm_score(E)
    assert want.dtype == dtype
    np.testing.assert_array_equal(got[:n_row, :n_col], want)
    assert np.all(got[:n_row, n_col:] == SENTINEL) and np.all(got[n_row] == SENTINEL)


# ---- xmve_count_before / xmve_count_band_f64 ----------------------------------------------------------------------
def test_count_before_with_ties_and_idx_offset(N):
    rng = np.random.default_rng(21)
    n_entries, cap, idx_offset = 300, 257, 5000
    exact = rng.integers(0, 6, (n_entries, cap)) * 0.125      # exact ties with s_gt everywhere
    idx = rng.integers(0, 10000, (n_entries, cap)).astype(np.int32)
    counts = rng.integers(0, cap + 100, n_entries).astype(np.int32)
    counts[:3] = [0, cap, cap + 1]
    s_gt = rng.integers(0, 6, n_entries) * 0.125
    g = rng.integers(idx_offset, idx_offset + 10000, n_entries).astype(np.int64)
    before0 = rng.integers(0, 1000, n_entries).astype(np.int64)
    for e in range(n_entries):
        exact[e, min(counts[e], cap):] = np.inf                # past the count: would be counted if read
    want = before0.copy()
    for e in range(n_entries):
        n = min(counts[e], cap)
        x, gid = exact[e, :n], idx[e, :n].astype(np.int64) + idx_offset
        want[e] += int(np.sum((x > s_gt[e]) | ((x == s_gt[e]) & (gid < g[e]))))
    exact_d = _buffer(exact, cap, np.inf, extra_rows=0)
    before = torch.from_numpy(before0).cuda()
    idx_d, counts_d, s_d, g_d = (torch.from_numpy(t).cuda() for t in (idx, counts, s_gt, g))
    N.call("xmve_count_before", N.ptr(exact_d), N.ptr(idx_d), N.ptr(counts_d), n_entries, cap, idx_offset, N.ptr(s_d),
           N.ptr(g_d), N.ptr(before), N.stream_ptr())
    assert np.array_equal(before.cpu().numpy(), want)


def test_count_band_f64_counts_past_the_band_cap(N):
    rng = np.random.default_rng(22)
    n_entries, cols, ld, band_cap = 5, 300000, 300003, 1000   # more columns than 64 blocks x 2048: the grid strides
    scores = rng.integers(0, 64, (n_entries, cols)) / 64.0
    scores[rng.random((n_entries, cols)) < 0.01] = np.nan     # never counted
    scores[4, :] = 0.5
    scores[4, rng.choice(cols, 300, replace=False)] = 0.75    # a band that fits: the list must be the whole band
    # delta = 0: the band is the exact ties of s_gt; delta = 0.02 spans one level either side
    s_gt = np.array([0.5, 0.5, 0.25, 1.5, 0.75])
    above0 = rng.integers(0, 100, n_entries).astype(np.int64)
    sc, s_d = _buffer(scores, ld, np.inf), torch.from_numpy(s_gt).cuda()
    bands = []
    for d in (0.0, 0.02):
        above = torch.from_numpy(above0).cuda()
        band_count = torch.zeros(n_entries, dtype=torch.int32, device="cuda")
        band_idx = torch.full((n_entries, band_cap), -1, dtype=torch.int32, device="cuda")
        N.call("xmve_count_band_f64", N.ptr(sc), n_entries, cols, ld, 0, N.ptr(s_d), d, N.ptr(above),
               N.ptr(band_count), N.ptr(band_idx), band_cap, N.stream_ptr())
        got_above, got_count, got_idx = above.cpu().numpy(), band_count.cpu().numpy(), band_idx.cpu().numpy()
        for e in range(n_entries):
            x = scores[e]
            hi, lo = s_gt[e] + d, s_gt[e] - d
            band = np.flatnonzero((x >= lo) & ~(x > hi))
            bands.append(band.size)
            assert got_above[e] == above0[e] + np.sum(x > hi), (d, e)
            assert got_count[e] == band.size, (d, e)          # keeps counting past band_cap
            listed = got_idx[e, :min(band.size, band_cap)]
            assert np.unique(listed).size == listed.size and np.all(np.isin(listed, band)), (d, e)
            if band.size <= band_cap:
                assert np.array_equal(np.sort(listed), band), (d, e)
            assert np.all(got_idx[e, min(band.size, band_cap):] == -1), (d, e)
    assert max(bands) > 3 * band_cap and 300 in bands and 0 in bands


def test_count_band_f64_refuses_more_than_65535_entries(N):
    """An argument check that returns before any launch: the small buffers are never touched."""
    buf = torch.zeros(16, dtype=torch.float64, device="cuda")
    cnt = torch.zeros(16, dtype=torch.int32, device="cuda")
    st = N.lib.xmve_count_band_f64(N.ptr(buf), 65536, 4, 4, 0, N.ptr(buf), 0.0, N.ptr(buf), N.ptr(cnt), N.ptr(cnt), 4,
                                   N.stream_ptr())
    assert st == -4                                                                          # XMVE_ERR_LIMIT
    torch.cuda.synchronize()
    assert bool((buf == 0).all()) and bool((cnt == 0).all())
