"""The oracle restatement against outputs of the reference itself (tests/golden, minted by
oracle/make_golden.py from /root/reference/LINAS-engine).  CPU only."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, case_inputs, load_golden
from oracle import linas

CASES = ["tiny_ragged", "small_cpv20", "c1_1k"]


def assert_blas_close(got, want, dtype, n_sum=1):
    """Dot products of unit rows in ``dtype`` (or a sum of ``n_sum`` of them) as the host BLAS summed them, against the
    reference's.  The goldens hold what the BLAS of the machine that minted them returned; another BLAS kernel or
    thread count adds in another order, which moves each such dot product by about one unit in the last place of 1.0
    (at most 1 eps over OpenBLAS's x86 kernels at 1, 3 and 8 threads) and a sum of n of them by about sqrt(n) units.
    The bound is 16 times that.  What is ranked or counted from these values is compared exactly."""
    eps = np.finfo(dtype).eps
    np.testing.assert_allclose(got, want, rtol=0, atol=16 * np.sqrt(n_sum) * eps)


def test_apscorer_known_answers():
    with open(os.path.join(GOLDEN, "apscorer.json")) as f:
        cases = json.load(f)
    assert len(cases) >= 20
    for c in cases:
        k = int(c["scorer"].split("@")[1]) if "@" in c["scorer"] else 0
        assert linas.ap_score(c["labels"], k) == c["score"], c


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("tag,cast", [("f32", np.float32), ("f64", np.float64)])
def test_full_path_matches_reference(manifest, name, tag, cast):
    V, Q, vid_ids, cap_ids, _ = case_inputs(manifest, name)
    g = load_golden(name)
    errors = linas.cal_error(V.astype(cast), Q.astype(cast))
    assert errors.dtype == cast
    assert_blas_close(errors[:8, :8], g["errors_head_" + tag], cast)
    assert_blas_close(errors.astype(np.float64).sum(), g["errors_sum_" + tag], cast, errors.size)
    v2t_gt, t2v_gt = linas.get_gt(vid_ids, cap_ids)
    np.testing.assert_array_equal(linas.gt_ranks(errors, t2v_gt), g["t2v_ranks_" + tag])
    np.testing.assert_array_equal(linas.gt_ranks(errors.T, v2t_gt), g["v2t_ranks_" + tag])
    perf = np.array(linas.cal_perf(errors, v2t_gt, t2v_gt), dtype=np.float64)
    np.testing.assert_array_equal(perf, g["perf_" + tag])       # bit-identical floats
    top10 = np.stack([linas.topk_ids(errors[i], 10) for i in range(min(64, len(errors)))])
    np.testing.assert_array_equal(top10, g["top10_" + tag])


def test_containers_and_elementwise(manifest):
    V, Q, vid_ids, cap_ids, _ = case_inputs(manifest, "tiny_ragged")
    rec, g = manifest["tiny_ragged"], load_golden("tiny_ragged")
    v2t_gt, t2v_gt = linas.get_gt(vid_ids, cap_ids)
    assert v2t_gt == rec["v2t_gt"]
    assert {str(k): v for k, v in t2v_gt.items()} == rec["t2v_gt"]
    assert list(t2v_gt.keys()) == [int(k) for k in rec["t2v_gt"].keys()]      # same insertion order
    assert any(len(x) == 0 for x in v2t_gt)                                   # ragged: empty rows exist
    for tag, cast in (("f32", np.float32), ("f64", np.float64)):
        Vc, Qc = V.astype(cast), Q.astype(cast)
        assert_blas_close(linas.cal_error(Vc, Qc), g["errors_" + tag], cast)
        assert_blas_close(linas.cal_simi(Qc, Vc), g["simi_" + tag], cast)
        np.testing.assert_array_equal(linas.norm_score(g["errors_" + tag]), g["norm_score_" + tag])
        np.testing.assert_array_equal(linas.l2norm(Vc), g["l2norm_" + tag])


def test_legacy_metrics(manifest):
    from cross_modal_video_engine_b200 import synth
    from conftest import input_sha256
    rec = manifest["legacy"]
    V, Q, _, _, _ = synth.msrvtt_like(rec["seed"], 40, 5, 48, 2.0)
    assert input_sha256(V, Q) == rec["input_sha256"]
    errors = linas.cal_error(V.astype(np.float64), Q.astype(np.float64))
    assert linas.t2v(errors, 5) == rec["t2v"]
    assert linas.v2t(errors, 5) == rec["v2t"]
    assert float(linas.t2v_inv_rank(errors, 5)) == rec["t2v_inv_rank"]
    assert float(linas.v2t_inv_rank(errors, 5)) == rec["v2t_inv_rank"]
    assert [float(x) for x in linas.v2t_inv_rank_multi(errors, 5)] == rec["v2t_inv_rank_multi"]


def test_multifusion_time_process_golden(manifest):
    import torch
    from cross_modal_video_engine_b200 import synth
    from oracle import multifusion
    if "unavailable" in manifest["mf_time_process"]:
        pytest.skip("reference combiner was not importable when goldens were minted")
    x = torch.from_numpy(synth.gaussian(31, 37 * 8, 640).reshape(37, 8, 640))
    np.testing.assert_array_equal(multifusion.time_process(x).numpy(), load_golden("mf_time_process")["pooled"])


# ---- MultiFusion: the restatement against the UNMODIFIED reference functions (oracle/make_golden_mf.py) ----------
def _mf_manifest():
    with open(os.path.join(GOLDEN, "mf_cirr.json")) as f:
        return json.load(f)


def mf_case_inputs(rec, n_query=None):
    from cross_modal_video_engine_b200 import synth
    from conftest import input_sha256
    out = synth.composed_retrieval(rec["seed"], rec["n_index"], n_query or rec["n_query"],
                                   frames=rec.get("frames", 8), sigma=rec.get("sigma", 0.5))
    return out


@pytest.mark.parametrize("name", ["a", "b", "c", "d"])
def test_multifusion_oracle_matches_reference_validate(name):
    """validate.compute_cirr_val_metrics (validate.py:27-143, unmodified) -> 7-tuple + results_wo_attn top-100."""
    import torch
    from conftest import input_sha256
    from oracle import multifusion
    rec = _mf_manifest()["cases"][name]
    index, P, names, ref, tgt = mf_case_inputs(rec)
    assert input_sha256(index, P, names, ref, tgt) == rec["input_sha256"], "synthetic generator drifted"
    metrics, top = multifusion.compute_cirr_val_metrics(torch.from_numpy(P), torch.from_numpy(index), names, ref, tgt)
    assert [float(x) for x in metrics] == rec["metrics"]                  # bit-identical floats
    np.testing.assert_array_equal(top, load_golden("mf_cirr_" + name)["top100"])


def test_multifusion_reference_cannot_take_a_multiple_of_32_queries():
    """Recorded quirk: the empty trailing block of validate.py:71 raises in reshape(0, -1) (:96-97)."""
    rec = _mf_manifest()["mult32"]
    assert rec["n_query"] % 32 == 0 and rec.get("raises") == "RuntimeError"


@pytest.mark.parametrize("name", ["i1", "i2"])
def test_multifusion_oracle_matches_reference_inference(name):
    """inference.compute_cirr_val_metrics (inference.py:26-66, unmodified) -> top-1 name."""
    import torch
    from conftest import input_sha256
    from oracle import multifusion
    rec = _mf_manifest()["inference"][name]
    index, P, names, _, _ = mf_case_inputs(rec, n_query=3)
    assert input_sha256(index, P, names) == rec["input_sha256"]
    pooled = torch.from_numpy(index).mean(dim=1)
    tar_list = ["vid_%d.mp4" % int(x) for x in names]
    got = [multifusion.top1_name(torch.from_numpy(P[i:i + 1]), pooled, tar_list) for i in range(3)]
    assert got == rec["top1"]


# ---- C1 with embeddings from the reference's random-init model (oracle/make_golden_c1_model.py) ------------------
def c1_model_inputs():
    g = load_golden("c1_model")
    vid, cap = g["vid"], load_golden("c1_model_cap")["cap"]          # two files: each stays under 1 MB
    n_v, per = len(vid), len(cap) // len(vid)
    video_ids = ["video%d" % i for i in range(n_v)]
    caption_ids = ["video%d#enc#%d" % (j // per, j % per) for j in range(len(cap))]
    return g, vid, cap, video_ids, caption_ids


def test_c1_random_init_model_embeddings_oracle():
    g, vid, cap, video_ids, caption_ids = c1_model_inputs()
    assert vid.dtype == np.float32 and vid.shape[1] == 1536
    np.testing.assert_allclose(np.linalg.norm(vid.astype(np.float64), axis=1), 1.0, atol=1e-6)   # Latent_mapping l2norm
    errors = linas.cal_error(vid.astype(np.float64), cap.astype(np.float64))
    assert_blas_close(errors[:6, :6], g["errors_head"], np.float64)
    assert_blas_close(errors.sum(), g["errors_sum"], np.float64, errors.size)
    v2t_gt, t2v_gt = linas.get_gt(video_ids, caption_ids)
    np.testing.assert_array_equal(np.array(linas.cal_perf(errors, v2t_gt, t2v_gt), dtype=np.float64), g["perf"])
    np.testing.assert_array_equal(linas.gt_ranks(errors, t2v_gt), g["t2v_ranks"])
    np.testing.assert_array_equal(np.stack([linas.topk_ids(errors[i], 10) for i in range(len(cap))]), g["top10"])
