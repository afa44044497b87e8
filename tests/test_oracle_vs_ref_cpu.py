"""Pins the oracle's NMS restatements -- and the library's host functions -- against the REFERENCE's OWN host code
({yolov8,yolov5}/src/postprocess.cpp and retinaface/common.hpp, compiled by oracle/Makefile with header shims for the
OpenCV / TensorRT includes those files pull in).  What that code returned on the inputs below is stored in
tests/golden/oracle_vs_ref.npz (tools/make_golden_vs_ref.py host): outputs as oracle.digest() strings, so every
comparison stays bit for bit, on any machine."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from tensorrtx_b200 import synth

GOLD = Path(__file__).resolve().parent / "golden" / "oracle_vs_ref.npz"


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _same(oracle, gold, key, mine):
    """`mine` is bit for bit what the reference's code returned (same rows, same order, same bits)."""
    return oracle.digest(mine) == str(gold[key])


@pytest.mark.parametrize("seed", range(4))
def test_v8_nms_equals_reference(oracle, gold, seed):
    heads = synth.yolov8_heads(2, seed=100 + seed)
    out, _ = oracle.yolov8_decode(heads)
    for b in range(2):
        mine, _ = oracle.nms(0, out[b], 1000, 90, 0.5, 0.45)
        key = f"v8_nms_{seed}_{b}"
        assert gold[key + "_n"] > 20
        assert _same(oracle, gold, key, mine)  # same rows, same order (class asc, conf desc), bit for bit


def _obb_plugin_rows(oracle, seed, B=2):
    heads = synth.yolov8_heads(B, seed=seed, nc=15, extra=1, n_obj=40)
    out, _ = oracle.yolov8_decode(heads, nc=15, is_obb=True)
    return out


@pytest.mark.parametrize("seed", range(3))
def test_v8_nms_obb_equals_reference(oracle, gold, seed):
    """nms_obb + probiou (mixed float/double C++ promotions): identical rows in identical order."""
    out = _obb_plugin_rows(oracle, 130 + seed)
    for b in range(out.shape[0]):
        for thr in (0.5, 0.2):
            mine, _ = oracle.nms(3, out[b], 1000, 90, 0.3, thr)
            key = f"v8_obb_{seed}_{b}_{thr}"
            assert gold[key + "_n"] > 10 and gold[key + "_n"] < int(out[b, 0])
            assert _same(oracle, gold, key, mine)


def test_v8_nms_ties_broken_by_bbox0_like_reference(oracle, gold):
    rng = np.random.default_rng(1)
    n = 400
    buf = np.zeros(1 + 1000 * 90, np.float32)
    rows = buf[1:1 + n * 90].reshape(n, 90)
    xy = rng.uniform(0, 600, (n, 2))
    wh = rng.uniform(10, 60, (n, 2))
    rows[:, :2], rows[:, 2:4] = xy, xy + wh
    rows[:, 4] = np.round(rng.uniform(0.5, 1.0, n), 2)  # many equal confidences, distinct bbox[0]
    rows[:, 5] = rng.integers(0, 3, n)
    buf[0] = n
    mine, _ = oracle.nms(0, buf, 1000, 90, 0.5, 0.45)
    assert _same(oracle, gold, "v8_ties", mine)


def test_v8_batch_nms_and_thresholds(oracle, gold):
    heads = synth.yolov8_heads(3, seed=7)
    out, _ = oracle.yolov8_decode(heads)
    for b in range(3):
        mine, _ = oracle.nms(0, out[b], 1000, 90, 0.3, 0.6)
        assert gold[f"v8_batch_{b}_n"] == len(mine) and _same(oracle, gold, f"v8_batch_{b}", mine)


@pytest.mark.parametrize("seed", range(3))
def test_v5_nms_equals_reference(oracle, gold, seed):
    heads = synth.yolov5_heads(1, seed=200 + seed, n_obj=200)
    out, _ = oracle.yolov5_decode(heads, synth.V5_ANCHORS)
    mine, _ = oracle.nms(1, out[0], 1000, 38, 0.5, 0.45)
    assert gold[f"v5_nms_{seed}_n"] > 50 and _same(oracle, gold, f"v5_nms_{seed}", mine)


@pytest.mark.parametrize("seed", range(3))
def test_retina_nms_equals_reference(oracle, gold, seed):
    heads = synth.retina_heads(1, seed=300 + seed, in_h=480, in_w=640, n_obj=60)
    out, _ = oracle.retina_decode(heads, in_h=480, in_w=640)
    tp = oracle.retina_total_priors(480, 640)
    mine, _ = oracle.nms(2, out[0], tp, 15, 0.1, 0.4)
    assert gold[f"retina_nms_{seed}_n"] > 20 and _same(oracle, gold, f"retina_nms_{seed}", mine)


def test_retina_conf_threshold_is_a_double_compare(oracle, gold):
    """`output[..] <= 0.1` compares against the DOUBLE 0.1: conf == 0.1f (> 0.1) is kept (common.hpp:113)."""
    tp = oracle.retina_total_priors(480, 640)
    buf = np.zeros(1 + tp * 15, np.float32)
    buf[0] = 3
    for i, c in enumerate([np.float32(0.1), np.nextafter(np.float32(0.1), np.float32(0)), np.float32(0.5)]):
        buf[1 + i * 15:1 + i * 15 + 4] = [100 * i, 0, 100 * i + 50, 50]
        buf[1 + i * 15 + 4] = c
    mine, _ = oracle.nms(2, buf, tp, 15, 0.1, 0.4)
    assert gold["retina_conf_n"] == 2 and _same(oracle, gold, "retina_conf", mine)


@pytest.mark.parametrize("variant,libname,fn", [(0, "libref_yolov8_host.so", "ref_v8_get_rect"),
                                                (1, "libref_yolov5_host.so", "ref_v5_get_rect")])
def test_get_rect_equals_reference(oracle, gold, variant, libname, fn):
    """get_rect (box in 640x640 network pixels -> cv::Rect in the original image): the reference's compiled host code vs
    the oracle vs the library's host function trtx_get_rect -- identical integers on 4000 boxes and 8 image sizes."""
    from tensorrtx_b200 import plugins as P
    rng = np.random.default_rng(50 + variant)
    rects = []
    for (w, h) in SIZES:
        for _ in range(500):
            if variant == 0:
                x1, y1 = rng.uniform(-30, 650, 2)
                bb = np.array([x1, y1, x1 + rng.uniform(-5, 400), y1 + rng.uniform(-5, 400)], np.float32)
            else:
                bb = np.array([rng.uniform(-30, 670), rng.uniform(-30, 670), rng.uniform(0, 500), rng.uniform(0, 500)], np.float32)
            r = oracle.get_rect(variant, w, h, bb)
            assert P.get_rect(w, h, bb, variant=variant) == tuple(int(v) for v in r)
            rects.append(r)
    assert _same(oracle, gold, fn, np.array(rects))   # fn of the reference's library libname


SIZES = ((1920, 1080), (1080, 1920), (640, 640), (1280, 720), (333, 777), (4000, 3000), (641, 640), (50, 60))


def test_get_rect_adapt_landmark_equals_reference(oracle, gold):
    """get_rect_adapt_landmark (yolov8/src/postprocess.cpp:38-69, pose models): box AND the 17 keypoints mapped back to the
    original image -- the library's host function against the reference's compiled code, identical integers and identical
    keypoint bits on 300 boxes x 8 image sizes."""
    from tensorrtx_b200 import plugins as P
    rng = np.random.default_rng(70)
    rects, lmks = [], []
    for (w, h) in SIZES:
        for _ in range(300):
            x1, y1 = rng.uniform(-30, 650, 2)
            bb = np.array([x1, y1, x1 + rng.uniform(-5, 400), y1 + rng.uniform(-5, 400)], np.float32)
            lmk = rng.uniform(-20, 660, 51).astype(np.float32)
            lmk[2::3] = rng.uniform(0, 1, 17).astype(np.float32)
            rect, mapped = P.get_rect_adapt_landmark(w, h, bb, lmk)
            rects.append(np.array(rect, np.int32)), lmks.append(np.asarray(mapped, np.float32))
    assert _same(oracle, gold, "v8_lmk_rects", np.array(rects))
    assert _same(oracle, gold, "v8_lmk", np.array(lmks))


def test_scale_mask_rect_and_process_decode_rows_equal_reference(gold):
    """scale_mask's crop of the 640x640 mask and its target size (postprocess.cpp:207-226; read back from the OpenCV shim) and
    process_decode_ptr_host (:131-147) -- the library's host functions against the reference's compiled code."""
    from tensorrtx_b200 import _lib as L
    lib = L.load()
    ref6 = iter(gold["scale_mask_rect"])
    for w in list(range(37, 2000, 97)) + [640, 641, 1920, 1080]:
        for h in (48, 479, 480, 640, 1080, 1920, 3000):
            r6, mine = next(ref6), (C.c_int * 4)()
            assert lib.trtx_scale_mask_rect(640, 640, w, h, mine) == 0
            assert list(mine) == r6[:4].tolist() and r6[4:].tolist() == [w, h]
    rng = np.random.default_rng(71)
    K = 200
    buf = np.zeros(1 + K * 7, np.float32)
    buf[0] = K
    rows = buf[1:].reshape(K, 7)
    rows[:, :6] = rng.uniform(0, 640, (K, 6)).astype(np.float32)
    rows[:, 6] = rng.integers(0, 2, K)
    out_ref, out_mine = gold["pdh"], np.zeros((K, 6), np.float32)
    n = lib.trtx_process_decode_ptr_host(buf.ctypes.data_as(C.POINTER(C.c_float)), 7, K, out_mine.ctypes.data_as(C.POINTER(C.c_float)))
    assert n == len(out_ref) == int(rows[:, 6].sum()) and np.array_equal(out_mine[:n], out_ref)


def test_process_decode_ptr_host_obb_equals_reference(gold):
    """process_decode_ptr_host_obb (yolov8/src/postprocess.cpp:273-290): kept rows of the oriented-box compact buffer (8-float rows,
    angle in column 7) -- the library's host function against the reference's compiled code."""
    from tensorrtx_b200 import _lib as L
    lib = L.load()
    rng = np.random.default_rng(72)
    for elem in (8, 9):
        K = 150
        buf = np.zeros(1 + K * elem, np.float32)
        buf[0] = K
        rows = buf[1:].reshape(K, elem)
        rows[:, :] = rng.uniform(-3, 640, (K, elem)).astype(np.float32)
        rows[:, 6] = rng.integers(0, 3, K)                  # keep flags 0, 1, 2: only == 1 is kept
        out_ref, out_mine = gold[f"pdh_obb_{elem}"], np.zeros((K, 7), np.float32)
        n = lib.trtx_process_decode_ptr_host_obb(buf.ctypes.data_as(C.POINTER(C.c_float)), elem, K, out_mine.ctypes.data_as(C.POINTER(C.c_float)))
        assert n == len(out_ref) == int((rows[:, 6] == 1).sum()) and n > 20 and np.array_equal(out_mine[:n], out_ref)
    assert lib.trtx_process_decode_ptr_host_obb(buf.ctypes.data_as(C.POINTER(C.c_float)), 7, K, out_mine.ctypes.data_as(C.POINTER(C.c_float))) < 0


def test_retina_get_rect_adapt_landmark_equals_reference(oracle, gold):
    """RetinaFace's get_rect_adapt_landmark (retinaface/common.hpp:65-89: box corners truncated to int, 5 landmark pairs mapped in
    place) -- the library's host function against the reference's compiled code: identical integers and landmark bits on 250 faces
    x 8 image sizes, for the 640x640 network of BASELINE config 3 and the 480x640 one the reference compiles in."""
    from tensorrtx_b200 import _lib as L
    lib = L.load()
    rng = np.random.default_rng(73)
    rects, lmks = [], []
    for (in_w, in_h) in ((640, 640), (640, 480)):
        for (w, h) in SIZES:
            for _ in range(250):
                x1, y1 = rng.uniform(-30, in_w + 10), rng.uniform(-30, in_h + 10)
                bb = np.array([x1, y1, x1 + rng.uniform(-5, 400), y1 + rng.uniform(-5, 400)], np.float32)
                lmk = rng.uniform(-20, 660, 10).astype(np.float32)
                l_mine, r_mine = lmk.copy(), (C.c_int * 4)()
                assert lib.trtx_retina_get_rect_adapt_landmark(in_w, in_h, w, h, bb.ctypes.data_as(C.POINTER(C.c_float)),
                                                               l_mine.ctypes.data_as(C.POINTER(C.c_float)), r_mine) == 0
                rects.append(np.array(list(r_mine), np.int32)), lmks.append(l_mine)
    assert _same(oracle, gold, "retina_lmk_rects", np.array(rects))
    assert _same(oracle, gold, "retina_lmk", np.array(lmks))
