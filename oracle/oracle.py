"""ctypes/numpy wrapper around oracle/libtrtx_oracle.so.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs.  Never imported by the product package (tensorrtx_b200/).
"""
from __future__ import annotations

import ctypes as C
import hashlib
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "libtrtx_oracle.so"
_lib = None

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB.exists() or LIB.stat().st_mtime < (HERE / "trtx_oracle.c").stat().st_mtime:
        subprocess.run(["make", "-C", str(HERE), str(LIB)], check=True, stdout=subprocess.DEVNULL)
    _lib = C.CDLL(str(LIB))
    return _lib


def digest(a) -> str:
    """sha256 of an array's dtype, shape and bytes: how golden files pin outputs that are compared bit for bit and are too
    large to store (tests/golden/*.npz)."""
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def sample_index(n: int, k: int = 64):
    """The rows of an n-row output that golden files keep when the output is compared with a tolerance and is too large
    to store whole: k of them (all when n <= k), ascending, fixed by n."""
    return np.sort(np.random.default_rng(n).choice(n, min(n, k), replace=False))


def _pp(arrs):
    a = (C.c_void_p * len(arrs))()
    for i, x in enumerate(arrs):
        assert x.dtype == np.float32 and x.flags["C_CONTIGUOUS"]
        a[i] = x.ctypes.data
    return a


def _ia(v):
    return (C.c_int * len(v))(*[int(x) for x in v])


def yolov8_decode(heads, strides=(8, 16, 32), net_w=640, net_h=640, nc=80, max_out=1000, det_floats=90, gate=0.1,
                  nk=17, kpt_thresh=0.0, is_seg=False, is_pose=False, is_obb=False):
    """-> (out [B, 1+max_out*det_floats] f32, anchor_idx [B, max_out] i32)."""
    lib = load()
    B = heads[0].shape[0]
    gh = [net_h // s for s in strides]
    gw = [net_w // s for s in strides]
    out = np.zeros((B, 1 + max_out * det_floats), np.float32)
    idx = np.full((B, max_out), -1, np.int32)
    lib.oracle_yolov8_decode(_pp(heads), B, len(heads), _ia(gh), _ia(gw), _ia(strides), nc, nk, C.c_float(kpt_thresh),
                             int(is_seg), int(is_pose), int(is_obb), max_out, det_floats, C.c_float(gate),
                             out.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p))
    return out, idx


def yolov5_decode(heads, anchors, strides=(8, 16, 32), net_w=640, net_h=640, nc=80, max_out=1000, det_floats=38,
                  ignore_thresh=0.1, is_seg=False):
    lib = load()
    B = heads[0].shape[0]
    gh = [net_h // s for s in strides]
    gw = [net_w // s for s in strides]
    anc = np.ascontiguousarray(np.asarray(anchors, np.float32).reshape(-1))
    out = np.zeros((B, 1 + max_out * det_floats), np.float32)
    idx = np.full((B, max_out), -1, np.int32)
    lib.oracle_yolov5_decode(_pp(heads), B, len(heads), _ia(gh), _ia(gw), anc.ctypes.data_as(C.c_void_p), nc, net_w,
                             net_h, int(is_seg), max_out, det_floats, C.c_float(ignore_thresh),
                             out.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p))
    return out, idx


def retina_total_priors(in_h, in_w):
    return sum((in_h // s) * (in_w // s) * 2 for s in (8, 16, 32))


def retina_decode(heads, in_h=640, in_w=640, gate=0.02):
    lib = load()
    B = heads[0].shape[0]
    tp = retina_total_priors(in_h, in_w)
    out = np.zeros((B, 1 + tp * 15), np.float32)
    idx = np.full((B, tp), -1, np.int32)
    lib.oracle_retina_decode(_pp(heads), B, in_h, in_w, C.c_double(gate), out.ctypes.data_as(C.c_void_p),
                             idx.ctypes.data_as(C.c_void_p))
    return out, idx


def yolov3_decode(heads, anchors, strides=(32, 16, 8), nc=80, max_out=1000, ignore_thresh=0.1):
    """heads: per level [B, 3*(5+nc), gh, gw] in the given level order.  -> (out [B, 1+max_out*7], anchor_idx [B, max_out])."""
    lib = load()
    B = heads[0].shape[0]
    gh = [h.shape[2] for h in heads]
    gw = [h.shape[3] for h in heads]
    flat = [np.ascontiguousarray(h.reshape(B, h.shape[1], -1), np.float32) for h in heads]
    anc = np.ascontiguousarray(np.asarray(anchors, np.float32).reshape(-1))
    out = np.zeros((B, 1 + max_out * 7), np.float32)
    idx = np.full((B, max_out), -1, np.int32)
    lib.oracle_yolov3_decode(_pp(flat), B, len(flat), _ia(gh), _ia(gw), _ia(strides), anc.ctypes.data_as(C.c_void_p), nc,
                             max_out, C.c_float(ignore_thresh), out.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p))
    return out, idx


def yolo26_gather(rows, nc=80, obb=False, max_out=300, det_floats=90, conf_thresh=0.4):
    """rows [B, A, 4+nc(+1)] -> (out [B, 1+max_out*det_floats], anchor_idx [B, max_out])."""
    lib = load()
    x = np.ascontiguousarray(rows, np.float32)
    B, A = x.shape[0], x.shape[1]
    out = np.zeros((B, 1 + max_out * det_floats), np.float32)
    idx = np.full((B, max_out), -1, np.int32)
    lib.oracle_yolo26_gather(x.ctypes.data_as(C.c_void_p), B, A, nc, int(obb), max_out, det_floats, C.c_float(conf_thresh),
                             out.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p))
    return out, idx


def anticov_decode(heads, in_h=640, in_w=640):
    lib = load()
    B = heads[0].shape[0]
    total = sum((in_h // s) * (in_w // s) * 2 for s in (8, 16, 32))
    out = np.zeros((B, 1 + total * 16), np.float32)
    idx = np.full((B, total), -1, np.int32)
    lib.oracle_anticov_decode(_pp(heads), B, in_h, in_w, out.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p))
    return out, idx


def nms(variant, plugin_out_img, max_rows, det_floats, conf_thresh, nms_thresh):
    """One image. variant 0 v8 / 1 v5 / 2 retinaface / 3 v8-obb (nms_obb, probiou). -> (res [n, det_floats], src_row [n])."""
    lib = load()
    lib.oracle_nms.restype = C.c_int
    p = np.ascontiguousarray(plugin_out_img, np.float32)
    res = np.zeros((max_rows, det_floats), np.float32)
    src = np.zeros(max_rows, np.int32)
    n = lib.oracle_nms(int(variant), p.ctypes.data_as(C.c_void_p), max_rows, det_floats, C.c_double(conf_thresh),
                       C.c_float(nms_thresh), res.ctypes.data_as(C.c_void_p), src.ctypes.data_as(C.c_void_p))
    return res[:n].copy(), src[:n].copy()


def cuda_decode_nms(plugin_out_img, max_rows, det_floats, conf_thresh, nms_thresh, max_objects):
    lib = load()
    p = np.ascontiguousarray(plugin_out_img, np.float32)
    out = np.zeros(1 + max_objects * 7, np.float32)
    lib.oracle_cuda_decode_nms(p.ctypes.data_as(C.c_void_p), max_rows, det_floats, C.c_float(conf_thresh),
                               C.c_float(nms_thresh), max_objects, out.ctypes.data_as(C.c_void_p))
    return out


def cuda_decode_nms_obb(plugin_out_img, max_rows, det_floats, conf_thresh, nms_thresh, max_objects):
    """decode_kernel_obb + nms_kernel_obb (one-shot, ProbIoU); rows of 8 floats (cx,cy,w,h,conf,cls,keep,angle)."""
    lib = load()
    p = np.ascontiguousarray(plugin_out_img, np.float32)
    out = np.zeros(1 + max_objects * 8, np.float32)
    lib.oracle_cuda_decode_nms_obb(p.ctypes.data_as(C.c_void_p), max_rows, det_floats, C.c_float(conf_thresh),
                                   C.c_float(nms_thresh), max_objects, out.ctypes.data_as(C.c_void_p))
    return out


def resize_bilinear(src, dh, dw):
    lib = load()
    s = np.ascontiguousarray(src, np.float32)
    dst = np.zeros((dh, dw), np.float32)
    lib.oracle_resize_bilinear(s.ctypes.data_as(C.c_void_p), s.shape[0], s.shape[1], dst.ctypes.data_as(C.c_void_p), dh, dw)
    return dst


def process_mask(variant, proto, bbox, coeffs, net_w=640, net_h=640):
    """variant 0 yolov8 / 1 yolov5; proto [nm, mh, mw]; -> mask [net_h, net_w] (process_mask of the seg drivers)."""
    lib = load()
    pr = np.ascontiguousarray(proto, np.float32)
    bb = np.ascontiguousarray(bbox, np.float32)
    cf = np.ascontiguousarray(coeffs, np.float32)
    out = np.zeros((net_h, net_w), np.float32)
    lib.oracle_process_mask(int(variant), pr.ctypes.data_as(C.c_void_p), pr.shape[0], pr.shape[1], pr.shape[2], net_w, net_h,
                            bb.ctypes.data_as(C.c_void_p), cf.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    return out


def roi_align(rois, feat, P, spatial_scale, sampling_ratio):
    """One image: rois [N,4], feat [C,H,W] -> [N,C,P,P] (RoIAlignForward, rcnn/RoiAlign.cu)."""
    lib = load()
    r = np.ascontiguousarray(rois, np.float32)
    f = np.ascontiguousarray(feat, np.float32)
    out = np.zeros((r.shape[0], f.shape[0], P, P), np.float32)
    lib.oracle_roi_align(r.ctypes.data_as(C.c_void_p), f.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                         r.shape[0], f.shape[0], f.shape[1], f.shape[2], P, C.c_float(spatial_scale), int(sampling_ratio))
    return out


def mask_rcnn_inference(indices, masks, out=None):
    """One image: indices [D] (float class ids), masks [D,nc,S,S] -> [D,S,S]."""
    lib = load()
    ind = np.ascontiguousarray(indices, np.float32)
    m = np.ascontiguousarray(masks, np.float32)
    D, nc, S, _ = m.shape
    out = np.zeros((D, S, S), np.float32) if out is None else np.ascontiguousarray(out, np.float32)
    lib.oracle_mask_rcnn_inference(ind.ctypes.data_as(C.c_void_p), m.ctypes.data_as(C.c_void_p),
                                   out.ctypes.data_as(C.c_void_p), D, S, nc)
    return out


def get_rect(variant, img_w, img_h, bbox, net_w=640, net_h=640):
    lib = load()
    b = np.ascontiguousarray(bbox, np.float32)
    r = np.zeros(4, np.int32)
    lib.oracle_get_rect(int(variant), net_w, net_h, img_w, img_h, b.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p))
    return r


def letterbox_matrix(sw, sh, dw, dh):
    lib = load()
    m = np.zeros(6, np.float32)
    lib.oracle_letterbox_matrix(sw, sh, dw, dh, m.ctypes.data_as(C.c_void_p))
    return m


def warpaffine(src_hwc_u8, dw, dh):
    lib = load()
    src = np.ascontiguousarray(src_hwc_u8, np.uint8)
    sh, sw = src.shape[:2]
    dst = np.zeros((3, dh, dw), np.float32)
    lib.oracle_warpaffine(src.ctypes.data_as(C.c_void_p), sw, sh, dst.ctypes.data_as(C.c_void_p), dw, dh)
    return dst


def rpn_decode(scores, deltas, image_h, image_w, stride, anchors, top_n):
    lib = load()
    B, A, H, W = scores.shape
    anchors = np.ascontiguousarray(anchors, np.float32)
    os_ = np.zeros((B, top_n), np.float32)
    ob = np.zeros((B, top_n, 4), np.float32)
    lib.oracle_rpn_decode(B, scores.ctypes.data_as(C.c_void_p), deltas.ctypes.data_as(C.c_void_p), H, W, image_h,
                          image_w, C.c_float(stride), anchors.ctypes.data_as(C.c_void_p), A, top_n,
                          os_.ctypes.data_as(C.c_void_p), ob.ctypes.data_as(C.c_void_p))
    return os_, ob


def rpn_nms(scores, boxes, post_nms_topk, nms_thresh):
    lib = load()
    B, pre = scores.shape
    ob = np.zeros((B, post_nms_topk, 4), np.float32)
    lib.oracle_rpn_nms(B, np.ascontiguousarray(scores).ctypes.data_as(C.c_void_p),
                       np.ascontiguousarray(boxes).ctypes.data_as(C.c_void_p), pre, post_nms_topk,
                       C.c_float(nms_thresh), ob.ctypes.data_as(C.c_void_p))
    return ob


def predictor_decode(scores, deltas, proposals, image_h, image_w, weights):
    lib = load()
    B, N, Cc = scores.shape
    w = np.ascontiguousarray(weights, np.float32)
    os_ = np.zeros((B, N), np.float32)
    ob = np.zeros((B, N, 4), np.float32)
    oc = np.zeros((B, N), np.float32)
    lib.oracle_predictor_decode(B, scores.ctypes.data_as(C.c_void_p), deltas.ctypes.data_as(C.c_void_p),
                                proposals.ctypes.data_as(C.c_void_p), N, Cc, image_h, image_w,
                                w.ctypes.data_as(C.c_void_p), os_.ctypes.data_as(C.c_void_p),
                                ob.ctypes.data_as(C.c_void_p), oc.ctypes.data_as(C.c_void_p))
    return os_, ob, oc


def batched_nms(method, scores, boxes, classes, detections_per_im, nms_thresh):
    lib = load()
    B, count = scores.shape
    os_ = np.zeros((B, detections_per_im), np.float32)
    ob = np.zeros((B, detections_per_im, 4), np.float32)
    oc = np.zeros((B, detections_per_im), np.float32)
    lib.oracle_batched_nms(int(method), B, np.ascontiguousarray(scores).ctypes.data_as(C.c_void_p),
                           np.ascontiguousarray(boxes).ctypes.data_as(C.c_void_p),
                           np.ascontiguousarray(classes).ctypes.data_as(C.c_void_p), count, detections_per_im,
                           C.c_float(nms_thresh), os_.ctypes.data_as(C.c_void_p), ob.ctypes.data_as(C.c_void_p),
                           oc.ctypes.data_as(C.c_void_p))
    return os_, ob, oc
