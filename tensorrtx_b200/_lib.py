"""ctypes binding of libtrtx_hot.so (the C ABI declared in include/trtx_hot.h).

There is NO fallback: if the shared library is missing or fails to load, importing the product
path raises.  The library is built in-tree by tensorrtx_b200/build.py (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

MAX_LEVELS = 8

OK, ERR_INVALID, ERR_WORKSPACE, ERR_CUDA, ERR_UNSUPPORTED = range(5)
YOLO_V8, YOLO_V5, YOLO_V3, YOLO_V26 = 0, 1, 2, 3
F32, F16 = 0, 1
BOX_LTRB, BOX_CXCYWH, BOX_RETINA, BOX_OBB = 0, 1, 2, 3
NMS_GREEDY, NMS_ONESHOT = 0, 1
ROI_WINDOW, ROI_DIRECT = 0, 1
RETINA_FACE, RETINA_ANTICOV = 0, 1

_ERR = {1: "TRTX_ERR_INVALID", 2: "TRTX_ERR_WORKSPACE", 3: "TRTX_ERR_CUDA", 4: "TRTX_ERR_UNSUPPORTED"}


class TrtxError(RuntimeError):
    pass


class YoloParams(C.Structure):
    _fields_ = [
        ("variant", C.c_int32),
        ("num_classes", C.c_int32),
        ("net_w", C.c_int32),
        ("net_h", C.c_int32),
        ("max_out", C.c_int32),
        ("det_floats", C.c_int32),
        ("num_levels", C.c_int32),
        ("grid_h", C.c_int32 * MAX_LEVELS),
        ("grid_w", C.c_int32 * MAX_LEVELS),
        ("strides", C.c_int32 * MAX_LEVELS),
        ("anchors", (C.c_float * 6) * MAX_LEVELS),
        ("is_seg", C.c_int32),
        ("is_pose", C.c_int32),
        ("is_obb", C.c_int32),
        ("num_kpts", C.c_int32),
        ("kpt_thresh", C.c_float),
        ("gate", C.c_float),
        ("in_dtype", C.c_int32),
        # per-call launch tuning (0 = default); the library holds no global knobs
        ("tune_class_slices", C.c_int32),
        ("tune_rows_in_flight", C.c_int32),
        ("tune_tma_pipeline", C.c_int32),
        ("tune_tma_stages", C.c_int32),
        ("tune_box_prefetch", C.c_int32),
        ("tune_nms_threads", C.c_int32),
    ]


class NmsParams(C.Structure):
    _fields_ = [
        ("box_format", C.c_int32),
        ("mode", C.c_int32),
        ("conf_thresh", C.c_float),
        ("nms_thresh", C.c_float),
        ("max_det", C.c_int32),
        ("class_aware", C.c_int32),
        ("tie_break_x0", C.c_int32),
        ("extra_floats", C.c_int32),
        ("extra_offset", C.c_int32),
    ]


class Gather(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("slots", C.c_int32), ("slot", C.c_int32),
                ("out_dev", C.c_void_p * 8), ("flags_dev", C.c_void_p * 8), ("ctrl_dev", C.c_void_p)]


class RetinaParams(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("gate", C.c_float), ("variant", C.c_int32)]


class ImageDesc(C.Structure):
    _fields_ = [
        ("data_dev", C.c_void_p),
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("pitch", C.c_int32),
        ("reserved", C.c_int32),
    ]


class MaskParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("variant", "net_w", "net_h", "mask_w", "mask_h", "num_coeffs", "row_floats",
                                         "coeff_offset", "max_masks")]


class RefineDetParams(C.Structure):
    _fields_ = [
        ("num_priors", C.c_int32),
        ("num_classes", C.c_int32),
        ("obj_thresh", C.c_float),
        ("conf_thresh", C.c_float),
        ("nms_thresh", C.c_float),
        ("top_k", C.c_int32),
        ("max_out", C.c_int32),
        ("variance", C.c_float * 2),
        ("reserved", C.c_int32),
    ]


REFINEDET_MAX_TOPK = 1024
REFINEDET_MAX_CLASSES = 91

# TRTX_LIB: another build of the same ABI (the probe build of tools/nms_probe.py); default = the in-tree release library
LIB_PATH = Path(os.environ.get("TRTX_LIB") or Path(__file__).resolve().parent / "lib" / "libtrtx_hot.so")

# every symbol include/trtx_hot.h declares: (name, restype, argtypes)
_vp, _sz, _i, _f = C.c_void_p, C.c_size_t, C.c_int, C.c_float
_pp = C.POINTER(C.c_void_p)
SYMBOLS = {
    "trtx_version": (C.c_char_p, []),
    "trtx_last_cuda_error": (_i, []),
    "trtx_yolo_params_init_v8": (_i, [C.POINTER(YoloParams), _i, _i, _i, _i, C.POINTER(C.c_int), _i]),
    "trtx_yolo_workspace_size": (_sz, [C.POINTER(YoloParams), _i]),
    "trtx_yolo_decode_enqueue": (_i, [C.POINTER(YoloParams), _i, _pp, _vp, _vp, _sz, _vp]),
    "trtx_nms_workspace_size": (_sz, [C.POINTER(NmsParams), _i, _i]),
    "trtx_nms_enqueue": (_i, [C.POINTER(NmsParams), _i, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "trtx_yolo_decode_nms_enqueue": (_i, [C.POINTER(YoloParams), C.POINTER(NmsParams), _i, _pp, _vp, _vp, _vp, _sz, _vp]),
    "trtx_yolo_scan_enqueue": (_i, [C.POINTER(YoloParams), _i, _pp, _vp, _sz, _vp]),
    "trtx_yolo_nms_after_scan_enqueue": (_i, [C.POINTER(YoloParams), C.POINTER(NmsParams), _i, _pp, _vp, _vp, _vp, _sz, _vp]),
    "trtx_retina_total_priors": (_i, [C.POINTER(RetinaParams)]),
    "trtx_retina_workspace_size": (_sz, [C.POINTER(RetinaParams), _i]),
    "trtx_retina_decode_enqueue": (_i, [C.POINTER(RetinaParams), _i, _pp, _vp, _vp, _sz, _vp]),
    "trtx_rpn_decode": (C.c_int64, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, C.POINTER(C.c_float), _i, _i, _vp, _sz, _vp]),
    "trtx_rpn_nms": (C.c_int64, [_i, _vp, _vp, _vp, _i, _i, _f, _vp, _sz, _vp]),
    "trtx_predictor_decode": (C.c_int64, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(C.c_float), _vp, _sz, _vp]),
    "trtx_batched_nms": (C.c_int64, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp, _sz, _vp]),
    "trtx_preprocess_batch_enqueue": (_i, [C.POINTER(ImageDesc), _i, _vp, _i, _i, _i, _vp]),
    "trtx_get_rect": (_i, [_i, _i, _i, _i, _i, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "trtx_roi_align": (_i, [_i, _vp, _vp, _vp, _i, C.c_float, _i, _i, _i, _i, _i, _vp]),
    "trtx_calib_letterbox_rect": (_i, [_i, _i, _i, _i, C.POINTER(C.c_int)]),
    "trtx_calib_letterbox_host": (_i, [_vp, _i, _i, C.c_size_t, _i, _i, _vp]),
    "trtx_roi_align_ex": (_i, [_i, _vp, _vp, _vp, _i, C.c_float, _i, _i, _i, _i, _i, _i, _vp]),
    "trtx_mask_rcnn_inference": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "trtx_process_mask_enqueue": (_i, [C.POINTER(MaskParams), _i, _vp, _vp, _i, _vp, _vp]),
    "trtx_letterbox_matrix": (None, [_i, _i, _i, _i, C.POINTER(C.c_float)]),
    "trtx_abi_sizeof": (_sz, [_i]),
    "trtx_get_rect_adapt_landmark": (_i, [_i, _i, _i, _i, C.POINTER(C.c_float), C.POINTER(C.c_float), _i, C.POINTER(C.c_int)]),
    "trtx_retina_get_rect_adapt_landmark": (_i, [_i, _i, _i, _i, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "trtx_process_decode_ptr_host": (_i, [C.POINTER(C.c_float), _i, _i, C.POINTER(C.c_float)]),
    "trtx_process_decode_ptr_host_obb": (_i, [C.POINTER(C.c_float), _i, _i, C.POINTER(C.c_float)]),
    "trtx_scale_mask_rect": (_i, [_i, _i, _i, _i, C.POINTER(C.c_int)]),
    "trtx_scale_mask_enqueue": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "trtx_yolo_decode_nms_gather_enqueue": (_i, [C.POINTER(YoloParams), C.POINTER(NmsParams), _i, _pp, _vp, _vp, _vp, _sz,
                                                 C.POINTER(Gather), _vp]),
    "trtx_gather_wait_enqueue": (_i, [C.POINTER(Gather), _vp]),
    "trtx_gather_push_enqueue": (_i, [C.POINTER(Gather), _vp, _i, _i, _i, _vp]),
    "trtx_gather_push_many_enqueue": (_i, [C.POINTER(Gather), _pp, _i, _i, _i, _i, _vp]),
    "trtx_gather_wait_many_enqueue": (_i, [C.POINTER(Gather), _i, _vp]),
    "trtx_peer_alloc": (_i, [_sz, C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]),
    "trtx_peer_open": (_i, [C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]),
    "trtx_peer_close": (_i, [_vp]),
    "trtx_peer_free": (_i, [_vp]),
    "trtx_refinedet_priors": (_i, [_i, _i, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                   C.POINTER(C.c_float), _vp]),
    "trtx_refinedet_workspace_size": (_sz, [C.POINTER(RefineDetParams), _i]),
    "trtx_refinedet_detect_enqueue": (_i, [C.POINTER(RefineDetParams), _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load libtrtx_hot.so; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise TrtxError(
            f"{LIB_PATH} is missing: build it with `python -m tensorrtx_b200.build` "
            "(or __graft_entry__.build()). There is no CPU/PyTorch fallback for this path."
        )
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    for which, st in enumerate((YoloParams, NmsParams, RetinaParams, ImageDesc, MaskParams, RefineDetParams)):
        if lib.trtx_abi_sizeof(which) != C.sizeof(st):
            raise TrtxError(f"{LIB_PATH} was built from a different trtx_hot.h: sizeof({st.__name__}) = "
                            f"{lib.trtx_abi_sizeof(which)} in the library, {C.sizeof(st)} in the binding (rebuild)")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        extra = ""
        if rc == ERR_CUDA:
            extra = f" (cudaError {load().trtx_last_cuda_error()})"
        raise TrtxError(f"{what} failed: {_ERR.get(rc, rc)}{extra}")


def ptr_array(ptrs) -> "C.Array":
    arr = (C.c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr
