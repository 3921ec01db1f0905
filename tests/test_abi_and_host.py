"""CPU-only checks: the C-ABI library loads and exports every symbol include/xmve.h declares (no compute
call without a GPU), compute entry points fail loudly without a device, and the host-side logic
(ground-truth containers, shard ranges, search plan, merge rule) is right."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, case_inputs
from oracle import linas


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "xmve.h")) as f:
        text = f.read()
    return sorted(set(re.findall(r"XMVE_API\s+(?:const\s+char\*|int64_t|int)\s+(xmve_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(os.path.join(ROOT, "cross-modal-video-engine_b200", "libxmve.so"))
    syms = _declared_symbols()
    assert len(syms) >= 16
    for s in syms:
        assert hasattr(lib, s), "libxmve.so does not export %s" % s
    assert lib.xmve_version() == 100


def test_binding_covers_the_header():
    from cross_modal_video_engine_b200 import _native
    assert set(_native.SIGNATURES) | {"xmve_last_error", "xmve_packed_topk_bytes"} == set(_declared_symbols())
    assert _native.lib.xmve_packed_topk_bytes(3, 5) == 256              # 3*5*16 + 3*4 = 252 -> padded to 16


def test_binding_argument_counts_match_the_header():
    """Every ctypes signature has as many arguments as the prototype in include/xmve.h (ABI drift guard)."""
    from cross_modal_video_engine_b200 import _native
    with open(os.path.join(ROOT, "include", "xmve.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    protos = dict(re.findall(r"XMVE_API\s+(?:const\s+char\*|int)\s+(xmve_\w+)\s*\(([^;]*?)\)\s*;", text, flags=re.S))
    for name, args in _native.SIGNATURES.items():
        params = protos[name].strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(args), "%s: header has %d parameters, the binding %d" % (name, n, len(args))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    from cross_modal_video_engine_b200 import _native, engine, evaluation, metrics, validate
    with pytest.raises(_native.XmveError):
        evaluation.cal_error(np.ones((2, 4)), np.ones((3, 4)))
    with pytest.raises(_native.XmveError):
        validate.cal_perf(np.zeros((2, 2)), [[0], [1]], {0: [0], 1: [1]})
    with pytest.raises(_native.XmveError):
        engine.CorpusStore(10, (8,))
    with pytest.raises(_native.XmveError):
        metrics.eval_q2m(np.zeros((2, 2)), [[0], [1]])
    lib = _native.lib                      # the C entry point itself refuses, too
    assert lib.xmve_device_check(-1) == -2
    assert b"no CPU path" in lib.xmve_last_error() or b"no GPU" in lib.xmve_last_error()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "cross-modal-video-engine_b200")
    seen = 0
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith(".py"):
                with open(os.path.join(dirpath, fn)) as f:
                    src = f.read()
                seen += 1
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), fn
    assert seen >= 15


def test_get_gt_matches_oracle_containers(manifest):
    from cross_modal_video_engine_b200 import metrics
    for name in ("tiny_ragged", "small_cpv20"):
        _, _, vid_ids, cap_ids, _ = case_inputs(manifest, name)
        ours, ref = metrics.get_gt(vid_ids, cap_ids), linas.get_gt(vid_ids, cap_ids)
        assert ours == ref and list(ours[1].keys()) == list(ref[1].keys())
    assert metrics.get_gt([], []) == ([], {})
    assert metrics.get_gt(["a"], []) == ([[]], {})
    assert metrics.get_gt(["a", "a"], ["a#1", "b#2", "a"]) == ([[0, 2], [0, 2]], {0: [0, 1], 2: [0, 1]})


def test_csr_and_median_helpers():
    from cross_modal_video_engine_b200 import metrics
    off, ids, mx = metrics._csr([[3, 1], [], [2]], 3)
    assert off.tolist() == [0, 2, 2, 3] and ids.tolist() == [3, 1, 2] and mx == 2
    with pytest.raises(KeyError):
        metrics._csr({0: [1]}, 2)          # a caption without a video: KeyError like util/metrics.py:142
    rng = np.random.default_rng(0)
    for n in (1, 2, 7, 8, 1001):
        ranks = rng.integers(1, 50, size=n).astype(np.int32)
        hist = np.bincount(ranks, minlength=52)
        assert metrics._median_from_hist(hist, n) == np.median(ranks)


def test_shard_range_partitions_exactly():
    from cross_modal_video_engine_b200 import distributed
    for n, w in ((10, 3), (1_080_000, 8), (7, 8), (0, 2)):
        spans = [distributed.shard_range(n, w, r) for r in range(w)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1


def test_merge_reference_rule():
    from cross_modal_video_engine_b200 import distributed
    s = torch.tensor([[[0.9, 0.5, float("-inf")]], [[0.9, 0.7, 0.1]]], dtype=torch.float64)
    i = torch.tensor([[[7, 3, -1]], [[2, 9, 4]]])
    ms, mi = distributed.merge_reference(s, i, 4)
    assert mi.tolist() == [[2, 7, 9, 3]] and ms.tolist() == [[0.9, 0.9, 0.7, 0.5]]


def test_search_plan_is_sane():
    from cross_modal_video_engine_b200 import engine
    store = engine.CorpusStore.__new__(engine.CorpusStore)
    for n, k in ((20000, 10), (1_000_000, 100), (10_000_000, 100), (1_080_000, 1000), (1_250_000, 101)):
        store.n = n
        p = store.plan(k)
        assert 1 <= p["step"] and p["n_sample"] * p["step"] >= n and p["n_sample"] <= n
        assert 1 <= p["j"] <= p["j_cap"] <= p["n_sample"]
        assert 2048 <= p["cap"] <= 32768 and p["j_cap"] * p["step"] <= p["cap"]
        assert p["n_sample"] <= 0.02 * n or n < 1_000_000     # the sampling pass stays a small fraction


def test_encode_vid_and_text_keep_the_reference_layout():
    """encode_vid / encode_text (evaluation.py:87-171) with a toy encoder and loader: rows scattered by dataset index,
    float64, ids in dataset order -- as one tensor on the encoder's device instead of a host array."""
    from cross_modal_video_engine_b200 import evaluation

    class DS:
        def __len__(self):
            return 7

    class Loader:
        dataset = DS()

        def __init__(self, with_support):
            self.with_support = with_support

        def __iter__(self):
            for idxs in ([4, 0, 6], [2, 5], [1, 3]):
                datas = torch.tensor([[float(i), 1.0] for i in idxs])
                ids = ["id%d" % i for i in idxs]
                yield (datas, datas * 2, idxs, ids) if self.with_support else (datas, idxs, ids)

    emb, ids = evaluation.encode_vid(lambda x: (x * 3).float(), Loader(False))
    assert emb.dtype == torch.float64 and ids == ["id%d" % i for i in range(7)]
    assert emb.tolist() == [[3.0 * i, 3.0] for i in range(7)]
    emb2 = evaluation.encode_text(lambda x, s: (x + s).float(), Loader(True), "GT", return_ids=False)
    assert emb2.tolist() == [[3.0 * i, 3.0] for i in range(7)]
    emb3, _ = evaluation.encode_text(lambda x: x.float(), Loader(False), "distill_from_best_model")
    assert emb3[:, 0].tolist() == [float(i) for i in range(7)]
    assert evaluation.encode_text(lambda x: x, Loader(False), "other") is None


def test_search_pipeline_two_level_sampling_on_cpu_model(monkeypatch):
    """The host pipeline on a CPU model of a shard (tests/cpu_model.py), at a size where the sampled threshold takes
    the two-level path (coarse floor + filter over the strided sample): one shard, and the same corpus cut into
    a large and a small shard (mixed sampling paths, global threshold) -- both must return the exact top-k."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpu_model
    from cross_modal_video_engine_b200 import engine
    cpu_model.patch_engine(monkeypatch.setattr)
    nv, nq, d, k = 2_200_000, 5, 16, 10
    g = torch.Generator().manual_seed(7)
    V, Q = torch.randn((nv, d), generator=g), torch.randn((nq, d), generator=g)
    assert (nv + engine.plan(k, nv)["step"] - 1) // engine.plan(k, nv)["step"] >= 16384      # two-level regime
    full = cpu_model.ModelShard(V, (d,))
    _, qr, qn, _, _ = full.prepare_queries(Q, [1.0])
    exact = full._exact(qr, qn, [1.0])
    ref = [cpu_model._sorted_topk(exact[r], torch.arange(nv), k) for r in range(nq)]
    stats = {}
    s, i = engine.search_shards([full], Q, k, stats=stats)
    assert all(torch.equal(i[r], ref[r][1]) for r in range(nq))
    assert all(torch.allclose(s[r], ref[r][0], rtol=0, atol=1e-12) for r in range(nq))
    assert 1e-3 < stats["eps"] < engine.EPS_X1
    cut = 2_150_000                                                 # big shard: two-level; small shard: plain sample
    shards = [cpu_model.ModelShard(V[:cut], (d,), 0), cpu_model.ModelShard(V[cut:], (d,), cut)]
    s2, i2 = engine.search_shards(shards, Q, k)
    assert all(torch.equal(i2[r], ref[r][1]) for r in range(nq))


@pytest.mark.parametrize("small_nv", [1000, 10 ** 9])
def test_search_rejects_exclude_shorter_than_the_batch(monkeypatch, small_nv):
    """``exclude`` holds one row per query: the selection, pilot and rescore kernels read ``excl[q]`` for every query,
    so a shorter one raises ValueError (as range_search does) instead of reaching them -- filtered and small path."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpu_model
    from cross_modal_video_engine_b200 import engine
    cpu_model.patch_engine(monkeypatch.setattr)
    g = torch.Generator().manual_seed(3)
    V, Q = torch.randn((20000, 16), generator=g), torch.randn((4, 16), generator=g)
    with pytest.raises(ValueError, match="exclude: expected one row"):
        engine.search_shards([cpu_model.ModelShard(V, (16,))], Q, 5, exclude=torch.tensor([3, -1]), small_nv=small_nv)
