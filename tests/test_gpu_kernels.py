"""Kernel-level parity tests (B200 only), each kernel called through the C ABI (ctypes) and compared with a
straightforward torch / NumPy statement of the same operation on the same seeded inputs."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def N():
    from cross_modal_video_engine_b200 import _native
    _native.require_device()
    return _native


def _rup(x, m):
    return (x + m - 1) // m * m


def _operands(N, nq, nv, d, seed, layout_q=0, layout_v=0):
    """Random raw rows -> bf16 operands via K1 (x1 or x3 layouts)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = torch.randn((nq, d), generator=g, device="cuda")
    v = torch.randn((nv, d), generator=g, device="cuda")
    dpad = _rup(d, 64)
    planes_q = 1 if layout_q == 0 else 3
    a = torch.zeros((_rup(nq, 128), planes_q * dpad), dtype=torch.bfloat16, device="cuda")
    b = torch.zeros((_rup(nv, 256), planes_q * dpad), dtype=torch.bfloat16, device="cuda")
    st = N.stream_ptr()
    N.call("xmve_prepare_rows", N.ptr(q), N.F32, nq, d, 1, d, None, 0, 0, None, None, N.ptr(a), a.stride(0), 0, layout_q, 1.0,
           0, st)
    N.call("xmve_prepare_rows", N.ptr(v), N.F32, nv, d, 1, d, None, 0, 0, None, None, N.ptr(b), b.stride(0), 0, layout_v, 1.0,
           0, st)
    return q, v, a, b


# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,frames,dtype", [(1000, 1536, 1, torch.float32), (77, 100, 1, torch.float64),
                                              (300, 640, 8, torch.float32), (5, 2048, 1, torch.float32),
                                              (130, 3000, 1, torch.float32), (64, 513, 2, torch.float32)])
def test_prepare_rows(N, n, d, frames, dtype):
    g = torch.Generator(device="cuda").manual_seed(1)
    shape = (n, d) if frames == 1 else (n, frames, d)
    x = (torch.randn(shape, generator=g, device="cuda") * 3).to(dtype)
    dpad = _rup(d, 64)
    op = torch.full((n, 3 * dpad + 64), 7.0, dtype=torch.bfloat16, device="cuda")
    raw = torch.zeros((n, d + 4), dtype=torch.float32, device="cuda")
    nrm = torch.zeros(n, dtype=torch.float64, device="cuda")
    res = torch.zeros(n, dtype=torch.float32, device="cuda")
    N.call("xmve_prepare_rows", N.ptr(x), N.F64 if dtype == torch.float64 else N.F32, n, d, frames, frames * d,
           N.ptr(raw), raw.stride(0), 4, N.ptr(nrm), N.ptr(res), N.ptr(op), op.stride(0), 64, N.OP_X3_CORPUS, 0.5, 0,
           N.stream_ptr())
    pooled = x.float() if frames == 1 else (x.float().sum(dim=1) / frames)
    ref_norm = torch.linalg.vector_norm(pooled.double(), dim=1)
    torch.testing.assert_close(raw[:, 4:4 + d], pooled, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(nrm, torch.linalg.vector_norm(raw[:, 4:4 + d].double(), dim=1), rtol=1e-13, atol=0)
    y = (0.5 * (raw[:, 4:4 + d].double() / nrm[:, None]).float())
    hi = y.to(torch.bfloat16)
    lo = (y - hi.float()).to(torch.bfloat16)
    assert torch.equal(op[:, 64:64 + d], hi)
    assert torch.equal(op[:, 64 + dpad:64 + dpad + d], lo)
    assert torch.equal(op[:, 64 + 2 * dpad:64 + 2 * dpad + d], hi)
    assert torch.all(op[:, :64] == 7.0)                       # columns before op_off untouched
    if dpad > d:
        assert torch.all(op[:, 64 + d:64 + dpad] == 0)        # zero-filled padding of each plane
    assert float((ref_norm - nrm).abs().max()) < 1e-4
    # measured quantisation residual of the hi plane: || 0.5 * x_hat - bf16(0.5 * x_hat) ||^2, rounded up
    exact = 0.5 * (raw[:, 4:4 + d].double() / nrm[:, None])
    ref_res = ((exact - hi.double()) ** 2).sum(1)
    # an upper bound by contract: exact on the generic path, inflated by 1e-3 on the register-resident fp32 path
    assert torch.all(res.double() >= ref_res * (1 - 1e-6)) and torch.all(res.double() <= ref_res * 1.0011 + 1e-30)
    assert torch.all(res.double().sqrt() <= 0.5 * 2.0 ** -8 * 1.0001)      # never above the worst-case rounding bound


SHAPES = [(1000, 1000, 1536), (77, 333, 100), (128, 256, 64), (129, 257, 192), (60, 70000, 2048), (513, 5000, 640)]


@pytest.mark.parametrize("tile", [6, 5, 4, 2, 1, 0])   # 2 wide pair 256x512 / 1 pair 256x256 / 0 single-CTA 128x256; 6 / 4 / 5 = the same with the dynamic unit scheduler
@pytest.mark.parametrize("nq,nv,d", SHAPES)
def test_score_store_matches_fp32_matmul_of_the_operands(N, nq, nv, d, tile, monkeypatch):
    monkeypatch.setenv("XMVE_TILE", str(tile))
    q, v, a, b = _operands(N, nq, nv, d, seed=nq + nv)
    out = torch.full((nq, nv), float("nan"), dtype=torch.float32, device="cuda")
    N.call("xmve_score_store", N.ptr(a), nq, a.stride(0), N.ptr(b), nv, b.stride(0), 1, a.shape[1], -1.0, N.ptr(out), nv,
           N.stream_ptr())
    torch.cuda.synchronize()
    ref = -(a[:nq].double() @ b[:nv].double().T)
    err = (out.double() - ref).abs().max().item()
    assert err < 2e-6, "tcgen05 tile mismatch: max abs err %g" % err      # fp32 accumulation of exact products


@pytest.mark.parametrize("nv,pad", [(1000, 24), (333, 5), (70, 2)])
def test_score_store_leaves_the_row_padding_alone(N, nv, pad):
    """Rows of the output are written through 128-byte segments staged in shared memory: columns >= nv of a padded
    output (out_ld > nv; aligned and unaligned leading dimensions) must keep the caller's bytes."""
    nq, d = 300, 256
    q, v, a, b = _operands(N, nq, nv, d, seed=11)
    out = torch.full((nq, nv + pad), -7.0, dtype=torch.float32, device="cuda")
    N.call("xmve_score_store", N.ptr(a), nq, a.stride(0), N.ptr(b), nv, b.stride(0), 1, a.shape[1], 1.0, N.ptr(out),
           out.stride(0), N.stream_ptr())
    ref = a[:nq].double() @ b[:nv].double().T
    assert float((out[:, :nv].double() - ref).abs().max()) < 2e-6
    assert bool((out[:, nv:] == -7.0).all())


@pytest.mark.parametrize("tile", [6, 4, 1])
def test_score_store_many_units_slow_epilogue(N, tile, monkeypatch):
    """20 000 x 2 990 x 4608 (the fp32 cal_error of the MSR-VTT shape): thousands of work units, many of them empty,
    and an epilogue that is busy storing -- the regime in which a mailbox hand-off with a too weak (CTA-scope)
    release let a peer-CTA warp read the next unit.  Every output element must be written, and right."""
    monkeypatch.setenv("XMVE_TILE", str(tile))
    nq, nv, k = 20000, 2990, 4608
    g = torch.Generator(device="cuda").manual_seed(1)
    a = torch.zeros((_rup(nq, 128), k), dtype=torch.bfloat16, device="cuda")
    b = torch.zeros((_rup(nv, 256), k), dtype=torch.bfloat16, device="cuda")
    a[:nq] = (torch.randn((nq, k), generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    b[:nv] = (torch.randn((nv, k), generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    for rep in range(3):
        out = torch.full((nq, nv), float("nan"), dtype=torch.float32, device="cuda")
        N.call("xmve_score_store", N.ptr(a), nq, a.stride(0), N.ptr(b), nv, b.stride(0), 1, k, -1.0, N.ptr(out), nv,
               N.stream_ptr())
        ref = -(a[:nq].float() @ b[:nv].float().T)
        assert not torch.isnan(out).any(), "rep %d: %d elements never written" % (rep, int(torch.isnan(out).sum()))
        assert float((out - ref).abs().max()) < 2e-4


def test_score_store_x3_split_reaches_fp32_accuracy(N):
    nq, nv, d = 700, 900, 1536
    q, v, a, b = _operands(N, nq, nv, d, seed=3, layout_q=N.OP_X3_QUERY, layout_v=N.OP_X3_CORPUS)
    out = torch.empty((nq, nv), dtype=torch.float32, device="cuda")
    N.call("xmve_score_store", N.ptr(a), nq, a.stride(0), N.ptr(b), nv, b.stride(0), 1, a.shape[1], 1.0, N.ptr(out), nv,
           N.stream_ptr())
    qn = q.double() / torch.linalg.vector_norm(q.double(), dim=1, keepdim=True)
    vn = v.double() / torch.linalg.vector_norm(v.double(), dim=1, keepdim=True)
    err = (out.double() - qn @ vn.T).abs().max().item()
    assert err < 3e-6, err


def test_score_store_strided_sample(N):
    nq, nv, d, step = 200, 10000, 256, 7
    q, v, a, b = _operands(N, nq, nv, d, seed=9)
    ns = (nv + step - 1) // step
    out = torch.empty((nq, ns), dtype=torch.float32, device="cuda")
    N.call("xmve_score_store", N.ptr(a), nq, a.stride(0), N.ptr(b), ns, b.stride(0), step, d, 1.0, N.ptr(out), ns,
           N.stream_ptr())
    ref = a[:nq].double() @ b[:nv:step].double().T
    assert (out.double() - ref).abs().max().item() < 2e-6


@pytest.mark.parametrize("tile", [6, 5, 4, 2, 1, 0])
@pytest.mark.parametrize("nq,nv,d,use_hi,quant", [(300, 50000, 512, False, 0.98), (77, 3000, 100, True, 0.98),
                                                  (1000, 200000, 128, False, 0.98),
                                                  # sparse windows: nearly every 32-column chunk that holds a candidate
                                                  # holds exactly one (the branch-free extraction), some hold two
                                                  (520, 60000, 640, False, 0.9985), (130, 40000, 192, True, 0.9985)])
def test_score_filter_window(N, nq, nv, d, use_hi, quant, tile, monkeypatch):
    monkeypatch.setenv("XMVE_TILE", str(tile))
    q, v, a, b = _operands(N, nq, nv, d, seed=11)
    s = (a[:nq].float() @ b[:nv].float().T)
    lo = torch.quantile(s[:, :2000], quant, dim=1).contiguous()
    hi = (lo + 0.05).contiguous() if use_hi else None
    cap = 8192
    cnt_above = torch.zeros(nq, dtype=torch.int32, device="cuda")
    cand_count = torch.zeros(nq, dtype=torch.int32, device="cuda")
    cand_score = torch.zeros((nq, cap), dtype=torch.float32, device="cuda")
    cand_idx = torch.full((nq, cap), -1, dtype=torch.int32, device="cuda")
    N.call("xmve_score_filter", N.ptr(a), nq, a.stride(0), N.ptr(b), nv, b.stride(0), 1, d if d % 64 == 0 else _rup(d, 64),
           N.ptr(lo), N.ptr(hi), N.ptr(cnt_above) if use_hi else None, N.ptr(cand_count), N.ptr(cand_score),
           N.ptr(cand_idx), cap, N.stream_ptr())
    torch.cuda.synchronize()
    margin = 2e-6                       # entries this close to a window edge may fall on either side
    inside = s > lo[:, None]
    if use_hi:
        above = s > hi[:, None]
        near = ((s - hi[:, None]).abs() < margin).sum(1)
        assert ((cnt_above - above.sum(1)).abs() <= near).all()
        inside = inside & ~above
    exp_count = inside.sum(1)
    near_lo = ((s - lo[:, None]).abs() < margin).sum(1) + (((s - hi[:, None]).abs() < margin).sum(1) if use_hi else 0)
    assert ((cand_count - exp_count).abs() <= near_lo).all()
    assert int(cand_count.max()) <= cap
    for r in range(0, nq, max(1, nq // 16)):
        n = int(cand_count[r])
        got = cand_idx[r, :n].long()
        assert len(set(got.tolist())) == n                                   # no duplicates
        torch.testing.assert_close(cand_score[r, :n], s[r, got], rtol=0, atol=2e-6)
        firm = (s[r] > lo[r] + margin) & ((s[r] < hi[r] - margin) if use_hi else True)
        assert set(torch.nonzero(firm).flatten().tolist()) <= set(got.tolist())


def test_score_filter_counts_past_cap(N):
    nq, nv, d = 64, 4000, 64
    q, v, a, b = _operands(N, nq, nv, d, seed=2)
    lo = torch.full((nq,), -10.0, device="cuda")
    cap = 128
    cand_count = torch.zeros(nq, dtype=torch.int32, device="cuda")
    cand_score = torch.zeros((nq, cap), dtype=torch.float32, device="cuda")
    cand_idx = torch.zeros((nq, cap), dtype=torch.int32, device="cuda")
    N.call("xmve_score_filter", N.ptr(a), nq, a.stride(0), N.ptr(b), nv, b.stride(0), 1, 64, N.ptr(lo), None, None,
           N.ptr(cand_count), N.ptr(cand_score), N.ptr(cand_idx), cap, N.stream_ptr())
    assert (cand_count == nv).all()                         # every (in-range) column counted, none of the padding


@pytest.mark.parametrize("rows,cols", [(50, 10000), (7, 33), (300, 70000)])
def test_row_kth(N, rows, cols):
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn((rows, cols), generator=g, device="cuda")
    x[0, : min(cols, 20)] = 1.25                            # ties
    counts = torch.randint(1, cols + 1, (rows,), generator=g, device="cuda", dtype=torch.int32)
    out = torch.empty(rows, device="cuda")
    j1, j2 = 3, 17
    out_dev = torch.empty(rows, device="cuda")
    half = torch.tensor([0.25], device="cuda")              # sub = 2 * sub_dev[0]: the device-side "2 eps"
    N.call("xmve_row_kth", N.ptr(x), rows, cols, cols, N.ptr(counts), j1, 0.5, None, j2, N.ptr(out), N.stream_ptr())
    N.call("xmve_row_kth", N.ptr(x), rows, cols, cols, N.ptr(counts), j1, 2.0, N.ptr(half), j2, N.ptr(out_dev),
           N.stream_ptr())
    assert torch.equal(out, out_dev)
    for r in range(rows):
        n = int(counts[r])
        srt = torch.sort(x[r, :n], descending=True).values
        a1 = srt[j1 - 1] - 0.5 if n >= j1 else torch.tensor(float("-inf"), device="cuda")
        a2 = srt[j2 - 1] if n >= j2 else torch.tensor(float("-inf"), device="cuda")
        assert out[r].item() == torch.maximum(a1, a2).item()


@pytest.mark.parametrize("rows,cols,j", [(40, 5000, 64), (9, 50, 101), (3, 3000, 1000)])
def test_row_topj(N, rows, cols, j):
    g = torch.Generator(device="cuda").manual_seed(15)
    x = torch.randn((rows, cols + 3), generator=g, device="cuda")
    x[0, :10] = 0.75                                         # ties
    counts = torch.randint(1, cols + 1, (rows,), generator=g, device="cuda", dtype=torch.int32)
    counts[-1] = cols
    out = torch.full((rows, j), 7.0, device="cuda")
    N.call("xmve_row_topj", N.ptr(x), rows, cols, x.stride(0), N.ptr(counts), j, N.ptr(out), N.stream_ptr())
    for r in range(rows):
        n = int(counts[r])
        ref = torch.sort(x[r, :n], descending=True).values[:j]
        assert torch.equal(out[r, :len(ref)], ref)
        assert torch.all(out[r, len(ref):] == float("-inf"))


def test_select_topk_and_merge(N):
    rows, cols, k = 40, 3000, 100
    g = torch.Generator(device="cuda").manual_seed(8)
    score = torch.randn((rows, cols), generator=g, device="cuda", dtype=torch.float64)
    score[:, ::7] = float("-inf")                           # not rescored
    score[3, 10:40] = 2.0                                   # exact ties -> index order
    idx = torch.stack([torch.randperm(100000, generator=g, device="cuda")[:cols] for _ in range(rows)]).int()
    counts = torch.full((rows,), cols - 5, dtype=torch.int32, device="cuda")
    excl = idx[:, 1].long() + 1000
    out_s = torch.empty((rows, k), dtype=torch.float64, device="cuda")
    out_i = torch.empty((rows, k), dtype=torch.int64, device="cuda")
    valid = torch.empty(rows, dtype=torch.int32, device="cuda")
    thr = torch.full((rows,), -1.0, device="cuda")
    cert = torch.empty(rows, dtype=torch.int32, device="cuda")
    nxt = torch.empty(rows, device="cuda")
    ten = torch.tensor([0.001], device="cuda")              # eps = 10 * eps_dev[0]
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    N.call("xmve_select_topk_i32", N.ptr(score), N.ptr(idx), rows, cols, N.ptr(counts), 1000, N.ptr(excl), k, N.ptr(thr),
           10.0, N.ptr(ten), None, N.ptr(out_s), N.ptr(out_i), N.ptr(valid), N.ptr(cert), N.ptr(nxt), N.ptr(n_bad),
           N.stream_ptr())
    assert int(n_bad) == 0
    for r in range(rows):
        s = score[r, :cols - 5].clone()
        i = idx[r, :cols - 5].long() + 1000
        keep = (s > float("-inf")) & (i != excl[r])
        s, i = s[keep], i[keep]
        order = sorted(range(len(s)), key=lambda t: (-s[t].item(), i[t].item()))[:k]
        assert out_i[r].tolist() == [i[t].item() for t in order]
        assert out_s[r].tolist() == [s[t].item() for t in order]
        assert int(valid[r]) == int(keep.sum())
        assert int(cert[r]) == 1 and abs(nxt[r].item() - (out_s[r, k - 1].item() - 0.01)) < 1e-5
    # K3 merge: split the winners over 4 "shards" and merge them back
    from cross_modal_video_engine_b200 import engine, distributed
    sh_s = torch.full((4, rows, k), float("-inf"), dtype=torch.float64, device="cuda")
    sh_i = torch.full((4, rows, k), -1, dtype=torch.int64, device="cuda")
    for gi in range(4):
        part_s, part_i = out_s[:, gi::4], out_i[:, gi::4]
        sh_s[gi, :, : part_s.shape[1]] = part_s
        sh_i[gi, :, : part_i.shape[1]] = part_i
    m_s, m_i = engine.merge_topk(sh_s, sh_i, k)
    assert torch.equal(m_s, out_s) and torch.equal(m_i, out_i)
    r_s, r_i = distributed.merge_reference(sh_s, sh_i, k)
    assert torch.equal(r_s, out_s) and torch.equal(r_i, out_i)
    # the same merge on PACKED per-rank blocks (what ONE all-gather delivers): [scores | rows | overflow flags]
    seg = engine.packed_bytes(rows, k)
    packed = torch.zeros((4, seg), dtype=torch.uint8, device="cuda")
    for gi in range(4):
        b_s, b_i, b_f = engine.packed_views(packed[gi], rows, k)
        b_s.copy_(sh_s[gi])
        b_i.copy_(sh_i[gi])
    engine.packed_views(packed[2], rows, k)[2][5] = 1       # shard 2 reports an overflowed list for row 5
    thr2 = torch.full((rows,), -1.0, device="cuda")
    thr2[7] = 10.0                                          # a threshold row 7's k-th score cannot clear
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    p_s, p_i, p_cert, p_nxt = engine._merge_packed(packed, rows, k, k, thr2, ten, n_bad)
    assert torch.equal(p_s, out_s) and torch.equal(p_i, out_i)
    want_cert = torch.ones(rows, dtype=torch.int32, device="cuda")
    want_cert[5] = 0
    want_cert[7] = 0
    assert torch.equal(p_cert, want_cert) and int(n_bad) == 2


def test_select_topk_more_valid_entries_than_the_sort_holds(N):
    """40 000 valid scores per row (the sort holds 16 384): the kernel first cuts at the k-th largest float-rounded
    score, which keeps a superset of the exact top-k -- including a block of exact ties across the k boundary."""
    rows, cols, k = 6, 40000, 100
    g = torch.Generator(device="cuda").manual_seed(18)
    score = torch.randn((rows, cols), generator=g, device="cuda", dtype=torch.float64)
    score[1] = 0.9 + 1e-9 * torch.randn(cols, generator=g, device="cuda", dtype=torch.float64)   # one float value
    score[2, 500:700] = 5.0                                                                     # 200 exact ties on top
    idx = torch.stack([torch.randperm(cols, generator=g, device="cuda") for _ in range(rows)]).int()
    counts = torch.full((rows,), cols, dtype=torch.int32, device="cuda")
    out_s = torch.empty((rows, k), dtype=torch.float64, device="cuda")
    out_i = torch.empty((rows, k), dtype=torch.int64, device="cuda")
    valid = torch.empty(rows, dtype=torch.int32, device="cuda")
    thr = torch.full((rows,), -10.0, device="cuda")
    cert = torch.empty(rows, dtype=torch.int32, device="cuda")
    nxt = torch.empty(rows, device="cuda")
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    N.call("xmve_select_topk_i32", N.ptr(score), N.ptr(idx), rows, cols, N.ptr(counts), 0, None, k, N.ptr(thr), 1e-3,
           None, None, N.ptr(out_s), N.ptr(out_i), N.ptr(valid), N.ptr(cert), N.ptr(nxt), N.ptr(n_bad), N.stream_ptr())
    assert (valid == cols).all() and int(n_bad) == 1
    for r in range(rows):
        if r == 1:                       # 40 000 scores that agree to float precision: reported as not certified
            assert int(cert[r]) == 0
            continue
        order = torch.argsort(idx[r].long(), stable=True)                  # index ascending ...
        s_sorted = score[r][order]
        top = torch.argsort(s_sorted, descending=True, stable=True)[:k]    # ... then score descending, stable
        assert torch.equal(out_s[r], s_sorted[top]) and torch.equal(out_i[r], idx[r].long()[order][top])
        assert int(cert[r]) == 1


def test_rescore_is_fp64_exact(N):
    """Two spaces, a bound and the two-round window.  Second case: the corpus norms sit in planes WIDER than the rows
    in use (a store filled below its capacity; the padding is NaN, so reading it shows), passed with their row stride
    as ``nv``, and a space width that is not a multiple of 4 (97 + 31), which takes the scalar fallback loop."""
    import ctypes as C
    nq, nv, cap = 33, 5000, 64
    for d0, pad in ((100, 0), (97, 37)):
        g = torch.Generator(device="cuda").manual_seed(4)
        q = torch.randn((nq, 128), generator=g, device="cuda")
        v = torch.randn((nv, 128), generator=g, device="cuda")
        qn = torch.stack([torch.linalg.vector_norm(q[:, :d0].double(), dim=1),
                          torch.linalg.vector_norm(q[:, d0:].double(), dim=1)])
        vn = torch.full((2, nv + pad), float("nan"), dtype=torch.float64, device="cuda")
        vn[0, :nv] = torch.linalg.vector_norm(v[:, :d0].double(), dim=1)
        vn[1, :nv] = torch.linalg.vector_norm(v[:, d0:].double(), dim=1)
        ld = vn.stride(0)
        idx = torch.randint(0, nv, (nq, cap), generator=g, device="cuda", dtype=torch.int32)
        approx = torch.randn((nq, cap), generator=g, device="cuda")
        count = torch.randint(0, cap + 20, (nq,), generator=g, device="cuda", dtype=torch.int32)
        bound = torch.zeros(nq, device="cuda")
        exact = torch.full((nq, cap), 123.0, dtype=torch.float64, device="cuda")
        off = (C.c_int32 * 3)(0, d0, 128)
        w = (C.c_double * 2)(0.7, 0.3)
        N.call("xmve_rescore", N.ptr(q), nq, 128, N.ptr(qn), N.ptr(v), ld, 128, N.ptr(vn), 2, off, w, 0, N.ptr(approx),
               N.ptr(idx), N.ptr(count), cap, N.ptr(bound), None, N.ptr(exact), N.stream_ptr())
        # two rounds give the same array: [0.5, inf) first, then [-0.3, 0.5) with the first round left untouched
        hi = torch.full((nq,), 0.5, device="cuda")
        lo = torch.full((nq,), -0.3, device="cuda")
        two = torch.full((nq, cap), 123.0, dtype=torch.float64, device="cuda")
        N.call("xmve_rescore", N.ptr(q), nq, 128, N.ptr(qn), N.ptr(v), ld, 128, N.ptr(vn), 2, off, w, 0, N.ptr(approx),
               N.ptr(idx), N.ptr(count), cap, N.ptr(hi), None, N.ptr(two), N.stream_ptr())
        first = two.clone()
        N.call("xmve_rescore", N.ptr(q), nq, 128, N.ptr(qn), N.ptr(v), ld, 128, N.ptr(vn), 2, off, w, 0, N.ptr(approx),
               N.ptr(idx), N.ptr(count), cap, N.ptr(lo), N.ptr(hi), N.ptr(two), N.stream_ptr())
        one = torch.full((nq, cap), 123.0, dtype=torch.float64, device="cuda")
        N.call("xmve_rescore", N.ptr(q), nq, 128, N.ptr(qn), N.ptr(v), ld, 128, N.ptr(vn), 2, off, w, 0, N.ptr(approx),
               N.ptr(idx), N.ptr(count), cap, N.ptr(lo), None, N.ptr(one), N.stream_ptr())
        assert torch.equal(two, one)
        assert torch.equal(two[approx >= 0.5], first[approx >= 0.5])
        for r in range(nq):
            n = min(int(count[r]), cap)
            rows = v[idx[r, :n].long()].double()
            s = 0.7 * (rows[:, :d0] @ q[r, :d0].double()) / (qn[0, r] * vn[0, idx[r, :n].long()]) \
                + 0.3 * (rows[:, d0:] @ q[r, d0:].double()) / (qn[1, r] * vn[1, idx[r, :n].long()])
            keep = approx[r, :n] >= 0
            assert torch.all(exact[r, :n][~keep] == float("-inf"))
            torch.testing.assert_close(exact[r, :n][keep], s[keep], rtol=0, atol=1e-14)
            assert torch.all(exact[r, n:] == 123.0)             # slots past the count are never written


def test_score_f64_and_normalize(N):
    nq, nv, d = 130, 257, 200
    g = torch.Generator(device="cuda").manual_seed(6)
    q = torch.randn((nq, d), generator=g, device="cuda", dtype=torch.float64)
    v = torch.randn((nv, d), generator=g, device="cuda")
    qn = torch.empty((nq, d), dtype=torch.float64, device="cuda")
    vn = torch.empty((nv, d), dtype=torch.float64, device="cuda")
    N.call("xmve_normalize_f64", N.ptr(q), N.F64, nq, d, d, N.ptr(qn), d, 0, N.stream_ptr())
    N.call("xmve_normalize_f64", N.ptr(v), N.F32, nv, d, d, N.ptr(vn), d, 0, N.stream_ptr())
    torch.testing.assert_close(qn, q / torch.linalg.vector_norm(q, dim=1, keepdim=True), rtol=0, atol=2e-16)
    out = torch.empty((nq, nv), dtype=torch.float64, device="cuda")
    N.call("xmve_score_f64", N.ptr(qn), nq, d, N.ptr(vn), nv, d, d, -1.0, N.ptr(out), nv, N.stream_ptr())
    torch.testing.assert_close(out, -(qn @ vn.T), rtol=0, atol=1e-14)


@pytest.mark.parametrize("j1,j2", [(1, 0), (10, 107), (200, 256), (257, 0), (60, 3000)])
def test_row_kth_pivot_and_radix_paths_agree_with_a_sort(N, j1, j2):
    """Small order statistics go through the pivot search (j <= 256), larger ones through the radix select; rows with
    heavy ties, -inf padding, a constant row, +inf / NaN entries and short rows must all give the exact statistic."""
    g = torch.Generator(device="cuda").manual_seed(41)
    rows, cols = 64, 9000
    x = 0.02 * torch.randn((rows, cols), generator=g, device="cuda") + 0.01
    x[1] = 0.5                                                # constant row
    x[2, ::2] = 0.125                                         # half of the row ties above everything else
    x[3, 300:] = float("-inf")                                # a padded union list: 300 finite values
    x[4, 5] = float("inf")
    x[5, 7] = float("nan")
    x[6] = torch.rand(cols, generator=g, device="cuda") ** 8  # heavy-tailed, far from Gaussian
    x[7] = -torch.rand(cols, generator=g, device="cuda") ** 8 # bulk at the TOP
    x[8, :50] = 3.0                                           # 50 exact ties on top of a Gaussian bulk
    counts = torch.full((rows,), cols, dtype=torch.int32, device="cuda")
    counts[9], counts[10], counts[11] = 700, 5, 0             # short rows
    out = torch.empty(rows, device="cuda")
    N.call("xmve_row_kth", N.ptr(x), rows, cols, cols, N.ptr(counts), j1, 0.0, None, j2, N.ptr(out), N.stream_ptr())
    for r in range(rows):
        if r == 5:
            continue                                          # NaN: ordering follows the float key (radix path); not asserted
        n = int(counts[r])
        srt = torch.sort(x[r, :n], descending=True).values
        a1 = srt[j1 - 1].item() if n >= j1 else float("-inf")
        a2 = srt[j2 - 1].item() if (j2 > 0 and n >= j2) else float("-inf")
        assert out[r].item() == max(a1, a2), (r, j1, j2)


# ---- rank / metric kernels ------------------------------------------------------------------------------
def _ap_reference(ranks, n_mem, k, first_only=False):
    """APScorer(k).score (basic/metric.py:25-46) from the 1-based ranks of the relevant entries."""
    length = k if 0 < k <= n_mem else n_mem
    if len(ranks) == 0:
        return 0.0
    if first_only:
        return 1.0 / ranks[0] if ranks[0] <= length else 0.0
    ap, hit = 0.0, 0
    for r in sorted(ranks):
        if r > length:
            break
        hit += 1
        ap += hit / r
    return ap / len(ranks)


@pytest.mark.parametrize("sizes", [[0, 1, 5, 33, 1000], [16384, 3], [16385, 7, 40000, 0, 2]])
def test_rank_metrics_any_list_length(N, sizes):
    """Per-query sort + reductions; lists of more than 16384 entries (ADVICE r1: they overran the shared buffer)
    are sorted in the global scratch.  Without the scratch the call must fail with XMVE_ERR_LIMIT."""
    from cross_modal_video_engine_b200 import metrics
    rng = np.random.default_rng(5)
    n_mem = 100000
    lists = [rng.permutation(n_mem)[:s] + 1 for s in sizes]
    off = np.zeros(len(sizes) + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    ranks = torch.from_numpy(np.concatenate(lists).astype(np.int32)).cuda()
    off_d = torch.from_numpy(off).cuda()
    for first_only, k in ((False, 0), (False, 1000), (True, 0)):
        best = torch.empty(len(sizes), dtype=torch.int32, device="cuda")
        ap = torch.empty(len(sizes), dtype=torch.float64, device="cuda")
        tallies = torch.zeros(4, dtype=torch.int64, device="cuda")
        hist = torch.zeros(n_mem + 2, dtype=torch.int32, device="cuda")
        metrics.rank_metrics(ranks, off_d, len(sizes), n_mem, first_only, k, max(sizes), best, ap, tallies, hist)
        want_best = [int(min(l)) if len(l) else n_mem + 1 for l in lists]
        assert best.cpu().tolist() == want_best
        assert ap.cpu().tolist() == [_ap_reference([int(x) for x in l], n_mem, k, first_only) for l in lists]
        assert tallies.cpu().tolist() == [sum(b <= t for b in want_best) for t in (1, 5, 10)] + [sum(want_best)]
        assert int(hist.sum()) == len(sizes)
    if max(sizes) > 16384:
        with pytest.raises(N.XmveError, match="sort_scratch"):
            N.call("xmve_rank_metrics", N.ptr(ranks), N.ptr(off_d), len(sizes), n_mem, 0, 0, max(sizes), None, None,
                   N.ptr(ap), None, None, None, N.stream_ptr())


def test_list_ranks(N):
    rng = np.random.default_rng(6)
    nq, kk, n_mem = 37, 1000, 50000
    lists = np.stack([rng.permutation(n_mem)[:kk] for _ in range(nq)]).astype(np.int64)
    lists[3, 500:] = -1                                                  # a padded list
    sizes = rng.integers(0, 40, nq)
    wanted = [np.concatenate([rng.choice(lists[q, :400], sizes[q] // 2, replace=False),
                              rng.integers(0, n_mem, sizes[q] - sizes[q] // 2)]) for q in range(nq)]
    off = np.zeros(nq + 1, np.int64)
    np.cumsum(sizes, out=off[1:])
    flat = np.concatenate(wanted).astype(np.int64)
    rank = torch.empty(len(flat), dtype=torch.int32, device="cuda")
    l_d, off_d, flat_d = torch.from_numpy(lists).cuda(), torch.from_numpy(off).cuda(), torch.from_numpy(flat).cuda()
    N.call("xmve_list_ranks", N.ptr(l_d), nq, kk, kk, N.ptr(off_d), N.ptr(flat_d), len(flat), n_mem + 1, N.ptr(rank),
           N.stream_ptr())
    want = []
    for q in range(nq):
        pos = {int(v): p + 1 for p, v in reversed(list(enumerate(lists[q]))) if v >= 0}
        want += [pos.get(int(w), n_mem + 1) for w in wanted[q]]
    assert rank.cpu().tolist() == want


def test_ap_at_k_with_a_huge_relevant_set(N):
    """avs.ap_at_k with 20 000 relevant shots for one query (> the 16384-entry shared sort)."""
    from cross_modal_video_engine_b200 import avs
    rng = np.random.default_rng(7)
    n_shots, kk = 200000, 1000
    idx = np.stack([rng.permutation(n_shots)[:kk] for _ in range(2)]).astype(np.int64)
    relevant = [np.concatenate([idx[0, ::3], rng.integers(0, n_shots, 20000)]), idx[1, :5]]
    relevant[0] = np.unique(relevant[0])
    ap, m = avs.ap_at_k(torch.from_numpy(idx).cuda(), relevant, n_shots, 1000)
    for q in range(2):
        pos = {int(v): p + 1 for p, v in enumerate(idx[q])}
        ranks = [pos.get(int(r), n_shots + 1) for r in relevant[q]]
        assert ap[q] == _ap_reference(ranks, n_shots, 1000)
    assert m == np.mean(ap)


# ---- two-round rescore: pilot kernels, device-side eps -------------------------------------------------------
def test_pilot_top_and_bound(N):
    from cross_modal_video_engine_b200 import engine
    g = torch.Generator(device="cuda").manual_seed(31)
    rows, cap, m, k, n_seg = 50, 700, 40, 100, 4
    lists = []
    for seg in range(n_seg):
        exact = torch.randn((rows, cap), generator=g, device="cuda", dtype=torch.float64)
        exact[torch.rand((rows, cap), generator=g, device="cuda") < 0.8] = float("-inf")     # not rescored
        exact[1] = float("-inf")                                                             # a row with no pilot at all
        idx = torch.stack([torch.randperm(5000, generator=g, device="cuda")[:cap] for _ in range(rows)]).int()
        counts = torch.randint(cap // 2, cap + 100, (rows,), generator=g, device="cuda", dtype=torch.int32)
        excl = idx[:, 3].long() + 7 * seg                                                    # an entry of every row
        out = torch.empty((rows, m), dtype=torch.float64, device="cuda")
        N.call("xmve_pilot_top", N.ptr(exact), N.ptr(idx), N.ptr(counts), rows, cap, 7 * seg, N.ptr(excl), m, N.ptr(out),
               N.stream_ptr())
        for r in range(rows):
            n = min(int(counts[r]), cap)
            keep = (exact[r, :n] > float("-inf")) & (idx[r, :n].long() + 7 * seg != excl[r])
            ref = torch.sort(exact[r, :n][keep], descending=True).values[:m]
            assert torch.equal(out[r, : len(ref)], ref) and torch.all(out[r, len(ref):] == float("-inf"))
        lists.append(out)
    union = torch.stack(lists)                                                               # [n_seg, rows, m]
    eps = torch.tensor([0.004], device="cuda")
    for kk in (1, 37, 100, 161):
        bound = engine._pilot_bound(union, kk, eps)
        for r in range(rows):
            allv = torch.sort(union[:, r, :].reshape(-1), descending=True).values
            if kk <= len(allv) and allv[kk - 1] > float("-inf"):
                want = allv[kk - 1].item() - float(eps)
                got = bound[r].item()
                assert got <= want and want - got < 1e-6 * max(1.0, abs(want))               # rounded DOWN to float
            else:
                assert bound[r].item() == float("-inf")


def test_eps_bound_matches_the_host_formula(N):
    import math
    from cross_modal_video_engine_b200 import engine
    g = torch.Generator(device="cuda").manual_seed(32)
    q_res = torch.rand((2, 5000), generator=g, device="cuda") * 3e-6
    dv2 = torch.tensor([2.9e-6], device="cuda")
    wts = [0.6, 0.4]
    got = float(engine._eps_device(q_res, dv2, wts, 2, 2048))
    want = engine.measured_eps(math.sqrt(float(q_res.sum(0).max())), math.sqrt(float(dv2)), wts, 2, 2048)
    assert want <= got <= want * (1 + 1e-6)                                                   # rounded UP to float
    q_res[1, 17] = float("nan")                                                               # a zero row: a-priori bound
    assert float(engine._eps_device(q_res, dv2, wts, 2, 2048)) == pytest.approx(engine.EPS_X1, rel=1e-6)
    assert float(engine._eps_device(q_res, dv2, wts, 2, 2048)) == engine.eps_fallback(wts, 2, 2048)
    assert engine.measured_eps(float("nan"), 1e-3, wts, 2, 2048) == engine.eps_fallback(wts, 2, 2048)
    q_res[1, 17] = 0.0
    dv2[0] = float("nan")                                                                     # a zero corpus row
    e_long = float(engine._eps_device(q_res, dv2, wts, 2, 6016))                             # past the constant
    assert e_long == engine.eps_fallback(wts, 2, 6016) > engine.EPS_X1


def test_select_topk_many_rows_use_the_small_sort(N):
    """>= 512 rows: the sort holds max(2048, 4k) entries; a row with more valid scores is cut at its k-th largest
    rounded score first and must still come out right and certified."""
    rows, cols, k = 600, 6000, 100
    g = torch.Generator(device="cuda").manual_seed(33)
    score = torch.randn((rows, cols), generator=g, device="cuda", dtype=torch.float64)
    score[:, 300:] = float("-inf")
    score[5] = torch.randn(cols, generator=g, device="cuda", dtype=torch.float64)             # 6000 valid entries
    idx = torch.stack([torch.randperm(cols, generator=g, device="cuda") for _ in range(rows)]).int()
    counts = torch.full((rows,), cols, dtype=torch.int32, device="cuda")
    out_s = torch.empty((rows, k), dtype=torch.float64, device="cuda")
    out_i = torch.empty((rows, k), dtype=torch.int64, device="cuda")
    thr = torch.full((rows,), -10.0, device="cuda")
    cert = torch.empty(rows, dtype=torch.int32, device="cuda")
    nxt = torch.empty(rows, device="cuda")
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    N.call("xmve_select_topk_i32", N.ptr(score), N.ptr(idx), rows, cols, N.ptr(counts), 0, None, k, N.ptr(thr), 1e-3,
           None, None, N.ptr(out_s), N.ptr(out_i), None, N.ptr(cert), N.ptr(nxt), N.ptr(n_bad), N.stream_ptr())
    assert int(n_bad) == 0 and bool((cert == 1).all())
    top_s, top_p = torch.topk(score, k, dim=1)
    assert torch.equal(out_s, top_s) and torch.equal(out_i, torch.gather(idx.long(), 1, top_p))


@pytest.mark.parametrize("rows", [600, 511])
def test_select_topk_reports_a_list_cut_by_float_ties(N, rows):
    """A shard's list before the merge (no threshold): row 7 holds 3 000 float-tied scores on top.  With 512 rows or
    more the sort holds max(2048, 4k) entries, so the kernel keeps an arbitrary 2 048 of the ties and must say so
    (cert = 0) for that row only; with 511 rows (the batches the engine re-runs such rows in) the sort holds them all
    and the list is the 100 smallest indices of the ties."""
    cols, k = 4096, 100
    g = torch.Generator(device="cuda").manual_seed(34)
    score = torch.randn((rows, cols), generator=g, device="cuda", dtype=torch.float64)
    score[:, 300:] = float("-inf")
    score[7] = torch.randn(cols, generator=g, device="cuda", dtype=torch.float64) - 5.0
    score[7, 500:3500] = 0.8                                                                    # 3 000 exact ties
    idx = torch.stack([torch.randperm(cols, generator=g, device="cuda") for _ in range(rows)]).int()
    counts = torch.full((rows,), cols, dtype=torch.int32, device="cuda")
    out_s = torch.empty((rows, k), dtype=torch.float64, device="cuda")
    out_i = torch.empty((rows, k), dtype=torch.int64, device="cuda")
    cert = torch.full((rows,), 7, dtype=torch.int32, device="cuda")
    n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
    N.call("xmve_select_topk_i32", N.ptr(score), N.ptr(idx), rows, cols, N.ptr(counts), 0, None, k, None, 0.0,
           None, None, N.ptr(out_s), N.ptr(out_i), None, N.ptr(cert), None, N.ptr(n_bad), N.stream_ptr())
    want = torch.ones(rows, dtype=torch.int32, device="cuda")
    if rows >= 512:
        want[7] = 0
    assert torch.equal(cert, want) and int(n_bad) == int((want == 0).sum())
    ids = idx.long()
    for r in range(rows):
        if int(want[r]) == 0:
            continue
        order = torch.argsort(ids[r], stable=True)                                 # index ascending ...
        top = torch.argsort(score[r][order], descending=True, stable=True)[:k]     # ... then score descending
        assert torch.equal(out_s[r], score[r][order][top]) and torch.equal(out_i[r], ids[r][order][top])
    if rows < 512:
        assert torch.equal(out_i[7], torch.sort(ids[7, 500:3500]).values[:k])
    with pytest.raises(N.XmveError, match="thr_next"):                            # a next threshold needs a threshold
        N.call("xmve_select_topk_i32", N.ptr(score), N.ptr(idx), rows, cols, N.ptr(counts), 0, None, k, None, 0.0,
               None, None, N.ptr(out_s), N.ptr(out_i), None, N.ptr(cert), N.ptr(torch.empty(rows, device="cuda")),
               None, N.stream_ptr())
