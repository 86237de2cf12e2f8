"""ctypes binding of libyolo_b200.so (include/yolo_b200.h).

The library is the product: there is no Python/torch fallback.  `lib()` raises if the shared
object has not been built (`python -c "import __graft_entry__ as g; g.build()"`), and every op in
`ops.py` raises if CUDA is not available.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int64, c_longlong,
                    c_size_t, c_ulonglong, c_void_p)

MAX_SCALES = 4
MAX_ANCHORS = 8
NMS_GRAPH, NMS_BITMASK = 0, 1
LAYOUT_BHWAC, LAYOUT_NCHW = 0, 1
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
MAP_MAX_T, MAP_MAX_GT = 16, 4096
MAP_BAD_CLASS, MAP_NMS_FAILED, MAP_INCONSISTENT = 1, 2, 4
COCO_MAX_A, COCO_MAX_M = 4, 4
LIB_NAME = "libyolo_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)


class LossDesc(Structure):
    """struct yb_loss_desc"""
    _fields_ = [
        ("S", c_int), ("B", c_int), ("B_global", c_longlong), ("A", c_int), ("nc", c_int),
        ("H", c_int * MAX_SCALES), ("W", c_int * MAX_SCALES),
        ("img_size", c_float), ("eps", c_float), ("w_box", c_float), ("w_cls", c_float),
        ("w_obj", c_float * MAX_SCALES), ("coef_box", c_float * MAX_SCALES),
        ("coef_obj", c_float * MAX_SCALES), ("coef_cls", c_float * MAX_SCALES),
        ("pred", c_void_p * MAX_SCALES), ("tgt", c_void_p * MAX_SCALES),
        ("anchors", c_void_p * MAX_SCALES), ("grad", c_void_p * MAX_SCALES),
        ("layout", c_int), ("dtype", c_int),
    ]


class HeadsDesc(Structure):
    """struct yb_heads_desc"""
    _fields_ = [
        ("S", c_int), ("B", c_int), ("A", c_int), ("nc", c_int),
        ("H", c_int * MAX_SCALES), ("W", c_int * MAX_SCALES), ("img_size", c_float),
        ("pred", c_void_p * MAX_SCALES), ("anchors", c_void_p * MAX_SCALES),
        ("layout", c_int), ("dtype", c_int),
    ]


# name -> (restype, argtypes); mirrors include/yolo_b200.h one to one
SIGNATURES = {
    "yb_version": (c_int, []),
    "yb_last_error": (c_char_p, []),
    "yb_launch_count": (c_ulonglong, []),
    "yb_timing_enable": (None, [c_int]),
    "yb_timing_collect": (c_int, [c_char_p, c_size_t]),
    "yb_decode_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "yb_decode_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "yb_decode_fwd_t": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                c_void_p]),
    "yb_decode_bwd_t": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                                c_int, c_void_p]),
    "yb_ciou_scratch_bytes": (c_size_t, [c_longlong]),
    "yb_ciou_fwd_bwd": (c_int, [c_void_p, c_void_p, c_longlong, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "yb_loss_workspace_bytes": (c_size_t, [POINTER(LossDesc)]),
    "yb_loss_partials": (c_int, [POINTER(LossDesc), c_void_p, c_void_p, c_size_t, c_void_p]),
    "yb_loss_finalize": (c_int, [POINTER(LossDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "yb_loss_sparse_workspace_bytes": (c_size_t, [POINTER(LossDesc), c_int]),
    "yb_loss_partials_sparse": (c_int, [POINTER(LossDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                        c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "yb_loss_grad_emit": (c_int, [POINTER(LossDesc), c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "yb_scale_inplace": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p]),
    "yb_anchor_iou": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "yb_build_targets": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_void_p), c_int, c_int, c_int,
                                 POINTER(c_int), c_int, c_int, c_int, c_void_p, c_void_p]),
    "yb_filter_workspace_bytes": (c_size_t, [POINTER(HeadsDesc)]),
    "yb_filter_compact": (c_int, [POINTER(HeadsDesc), c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_void_p, c_size_t, c_void_p]),
    "yb_filter_multilabel_workspace_bytes": (c_size_t, [POINTER(HeadsDesc), c_int]),
    "yb_filter_multilabel": (c_int, [POINTER(HeadsDesc), c_float, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "yb_nms_workspace_bytes": (c_size_t, [c_int, c_int]),
    "yb_nms_min_workspace_bytes": (c_size_t, [c_int, c_int]),
    "yb_nms_graph_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "yb_batched_nms": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_longlong, c_int,
                               c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "yb_nms_graph_stats": (c_int, [c_void_p, c_size_t, c_int, c_int, POINTER(c_ulonglong), POINTER(c_ulonglong),
                                   POINTER(c_ulonglong), c_void_p]),
    "yb_eval_counts": (c_int, [POINTER(HeadsDesc), POINTER(c_void_p), c_double, c_double, c_void_p, c_void_p]),
    "yb_selftest_sigmoid": (c_int, [POINTER(c_ulonglong), c_void_p]),
    "yb_pack_detections": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p]),
    "yb_map_match": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                             c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "yb_map_workspace_bytes": (c_size_t, [c_longlong, c_longlong, c_int]),
    "yb_map_precision": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                                 c_void_p, c_size_t, c_void_p, c_void_p]),
    "yb_coco_match": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p,
                              c_void_p, c_int, c_int, c_void_p, c_int, POINTER(c_double), c_int, c_void_p, c_void_p,
                              c_void_p, c_void_p]),
    "yb_coco_precision": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, POINTER(c_int),
                                  c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "yb_report_match": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_double, c_double,
                                c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
}

_lib = None


def lib():
    """The loaded library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this path.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().yb_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
