"""ctypes binding of ``libxmve.so`` (the C ABI declared in ``include/xmve.h``).

There is no fallback: if the shared library is missing the import fails with build instructions,
and every compute entry point fails loudly on a machine without an sm_100 GPU
(``XMVE_ERR_DEVICE``).  The oracle under ``oracle/`` is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxmve.so")

F32, F64 = 0, 1
OP_X1, OP_X3_QUERY, OP_X3_CORPUS = 0, 1, 2
NORM_PLAIN, NORM_EPS = 0, 1
MEASURE_L1, MEASURE_L2, MEASURE_JACCARD, MEASURE_SQL2, MEASURE_DOT, MEASURE_ORDER = 0, 1, 2, 3, 4, 5


class XmveError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "libxmve.so is not built (%s). Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "or `make -C cross-modal-video-engine_b200/csrc`. There is no CPU / PyTorch fallback." % LIB_PATH)

import torch  # noqa: E402,F401  -- loads libcudart.so.12 into the process; libxmve.so links the runtime shared

lib = C.CDLL(LIB_PATH)

_p, _i, _l, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
_i32 = C.c_int32

# name -> argtypes, in the order of include/xmve.h
SIGNATURES = {
    "xmve_version": [],
    "xmve_device_check": [_i],
    "xmve_sm_count": [],
    "xmve_prepare_rows": [_p, _i, _l, _i, _i, _l, _p, _l, _l, _p, _p, _p, _l, _l, _i, _f, _i, _p],
    "xmve_score_store": [_p, _l, _l, _p, _l, _l, _l, _i, _f, _p, _l, _p],
    "xmve_score_filter": [_p, _l, _l, _p, _l, _l, _l, _i, _p, _p, _p, _p, _p, _p, _i32, _p],
    "xmve_score_filter_labeled": [_p, _l, _l, _p, _l, _l, _l, _i, _p, _p, _p, _p, _p, _p, _i32, _p, _p, _p],
    "xmve_mask_scores": [_p, _i, _l, _l, _l, _p, _l, _p, _p],
    "xmve_row_kth": [_p, _l, _l, _l, _p, _i32, _f, _p, _i32, _p, _p],
    "xmve_rescore": [_p, _l, _l, _p, _p, _l, _l, _p, _i, _p, _p, _i, _p, _p, _p, _i32, _p, _p, _p, _p],
    "xmve_pilot_top": [_p, _p, _p, _l, _i32, _l, _p, _i32, _p, _p],
    "xmve_pilot_bound": [_p, _i32, _l, _i32, _i32, _f, _p, _p, _p],
    "xmve_eps_bound": [_p, _i32, _l, _p, _d, _i32, _f, _p, _p],
    "xmve_select_topk_i32": [_p, _p, _l, _l, _p, _l, _p, _i32, _p, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "xmve_select_topk_i64": [_p, _p, _l, _l, _p, _i32, _p, _f, _p, _p, _p, _p, _p, _p, _p, _p, _p],
    "xmve_merge_topk_packed": [_p, _i32, _l, _l, _i32, _p, _i32, _p, _f, _p, _p, _p, _p, _p, _p, _p],
    "xmve_range_select": [_p, _p, _p, _l, _i32, _l, _p, _p, _p, _p, _l, _p, _p, _p, _p],
    "xmve_pair_select": [_p, _p, _p, _l, _i32, _l, _p, _p, _p, _p, _l, _p, _p, _p, _p, _p],
    "xmve_range_merge": [_p, _p, _i32, _p, _l, _p, _l, _p, _p, _p],
    "xmve_row_topj": [_p, _l, _l, _l, _p, _i32, _p, _p],
    "xmve_normalize_f64": [_p, _i, _l, _i, _l, _p, _l, _i, _p],
    "xmve_score_f64": [_p, _l, _l, _p, _l, _l, _i, _d, _p, _l, _p],
    "xmve_score_f64_fused": [_p, _l, _l, _p, _l, _l, _i, _d, _d, _i, _p, _l, _p],
    "xmve_pairwise_f64": [_p, _l, _l, _p, _l, _l, _i, _i, _d, _d, _p, _l, _p],
    "xmve_triplet_cost": [_p, _l, _l, _d, _i, _p, _p],
    "xmve_gt_ranks": [_p, _i, _l, _l, _l, _i, _p, _p, _l, _l, _i32, _p, _p],
    "xmve_rank_metrics": [_p, _p, _l, _l, _i, _i, _i32, _p, _p, _p, _p, _p, _p, _p],
    "xmve_list_ranks": [_p, _l, _l, _l, _p, _p, _l, _i32, _p, _p],
    "xmve_count_before": [_p, _p, _p, _l, _i32, _l, _p, _p, _p, _p],
    "xmve_count_band_f64": [_p, _l, _l, _l, _l, _p, _d, _p, _p, _p, _i32, _p],
    "xmve_norm_score": [_p, _i, _l, _l, _l, _p, _l, _p, _p],
    "xmve_fuse_accumulate": [_p, _l, _p, _l, _i, _l, _l, _d, _i, _p],
}
for _name, _args in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.argtypes = _args
    _fn.restype = _i
lib.xmve_packed_topk_bytes.argtypes = [_l, _i32]
lib.xmve_packed_topk_bytes.restype = C.c_int64
lib.xmve_last_error.argtypes = []
lib.xmve_last_error.restype = C.c_char_p

#: number of kernel launches issued through this binding (bench.py reports it as gpu_launches)
launch_count = 0
_LAUNCHES = {"xmve_prepare_rows": 1, "xmve_score_store": 1, "xmve_score_filter": 1, "xmve_score_filter_labeled": 1, "xmve_mask_scores": 1,
             "xmve_row_kth": 1,
             "xmve_rescore": 1, "xmve_pilot_top": 1, "xmve_pilot_bound": 1, "xmve_eps_bound": 1, "xmve_merge_topk_packed": 1, "xmve_select_topk_i32": 1, "xmve_select_topk_i64": 1, "xmve_range_select": 1, "xmve_pair_select": 1, "xmve_range_merge": 1, "xmve_row_topj": 1, "xmve_normalize_f64": 1,
             "xmve_score_f64": 1, "xmve_score_f64_fused": 1, "xmve_pairwise_f64": 1, "xmve_triplet_cost": 1, "xmve_gt_ranks": 2, "xmve_rank_metrics": 1, "xmve_list_ranks": 1, "xmve_count_before": 1, "xmve_count_band_f64": 1, "xmve_norm_score": 3, "xmve_fuse_accumulate": 1}


def call(name, *args):
    """Call a C-ABI entry point; raise :class:`XmveError` with the library's message on failure."""
    global launch_count
    status = getattr(lib, name)(*args)
    if status != 0:
        raise XmveError("%s failed (%d): %s" % (name, status, lib.xmve_last_error().decode("utf-8", "replace")))
    launch_count += _LAUNCHES.get(name, 0)
    return status


def ptr(t):
    """Device pointer of a CUDA tensor (``None`` -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise XmveError("expected a CUDA tensor; libxmve has no CPU path")
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_device():
    """Fail loudly unless the current CUDA device is sm_100."""
    import torch
    if not torch.cuda.is_available():
        raise XmveError("no CUDA device: this engine runs hand-written sm_100a kernels only (no CPU fallback)")
    call("xmve_device_check", -1)
