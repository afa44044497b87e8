"""SURVEY 8f rank 4 + row a2: the older / other plugin variants through the same scan / pack / NMS kernels, each against
(1) the REFERENCE'S OWN plugin (compiled by oracle/Makefile and run on a B200 on the same inputs; what it returned is stored
in tests/golden/ref_kernels.npz, tools/make_golden_vs_ref.py device) and (2) the CPU oracle:
  yolov7   6-float Detection rows            yolov7/plugin/yololayer.cu:152-200, yolov7/include/types.h:11-16
  yolov3   exp-wh, dual confidence, 7 floats yolov3-spp/yololayer.cu:148-191
  yolo26   NMS-free gatherKernel, AoS input  yolo26/plugin/yololayer.cu:178-245
  retinafaceAntiCov  16-float rows           retinafaceAntiCov/decode.cu:110-172
The references' slot order is atomicAdd arrival: rows are compared as canonically sorted sets."""
from pathlib import Path

import numpy as np
import pytest
import torch

from tensorrtx_b200 import _lib as L
from tensorrtx_b200 import plugins as P
from tensorrtx_b200 import synth

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).resolve().parent / "golden" / "ref_kernels.npz"
ATOL = 1e-4
V3_ANCHORS = [k.anchors for k in P.YOLOV3_KERNELS]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _canon(rows):
    return rows[np.lexsort(tuple(rows[:, k] for k in range(rows.shape[1] - 1, -1, -1)))]


def _rows(buf, b, F, n=None):
    n = int(buf[b, 0]) if n is None else n
    return buf[b, 1:1 + n * F].reshape(n, F)


# ------------------------------------------------------------------ yolov7: 6-float rows -----------------
def _v7_kernels():
    return [P.YoloKernel(640 // s, 640 // s, a) for s, a in zip((8, 16, 32), synth.V5_ANCHORS)]


def test_yolov7_6_float_rows_vs_reference_kernel_and_oracle(oracle, dev, gold):
    B = 3
    heads = synth.yolov5_heads(B, seed=610)
    hd = [torch.from_numpy(h).to(dev) for h in heads]
    plug = P.YoloLayerPluginV7(80, 640, 640, 1000, _v7_kernels())
    out = torch.full((B, plug.output_elems()), -5.0, dtype=torch.float32, device=dev)
    ws = torch.empty(plug.getWorkspaceSize(B), dtype=torch.uint8, device=dev)
    assert plug.enqueue(B, hd, [out], ws) == 0
    got = out.cpu().numpy()
    orc, _ = oracle.yolov5_decode(heads, synth.V5_ANCHORS, det_floats=6)
    assert np.array_equal(gold["v7_counts"], got[:, 0]) and np.array_equal(orc[:, 0], got[:, 0]) and got[:, 0].min() > 100
    for b in range(B):
        g = _canon(_rows(got, b, 6))   # against the oracle.sample_index() rows of the reference's canonically sorted rows
        np.testing.assert_allclose(g[oracle.sample_index(len(g))], gold[f"v7_{b}"], rtol=3e-7, atol=0)  # FMA contraction
        np.testing.assert_allclose(_rows(got, b, 6), _rows(orc, b, 6), atol=ATOL, rtol=2e-6)                  # anchor order
        assert np.all(got[b, 1 + int(got[b, 0]) * 6:] == -5.0)   # nothing written past the rows
    # serialization layout of yolov7/plugin/yololayer.cu:62-77 round-trips
    q = P.YoloLayerPluginV7.deserialize(plug.serialize())
    assert q.serialize() == plug.serialize() and len(plug.serialize()) == plug.getSerializationSize()


# ------------------------------------------------------------------ yolov3 / v3-spp / v4 -----------------
@pytest.mark.parametrize("net,B", [((608, 608), 2), ((416, 352), 3)])
def test_yolov3_vs_reference_kernel_and_oracle(oracle, dev, gold, net, B):
    heads = synth.yolov3_heads(B, seed=620 + B, net_w=net[0], net_h=net[1])
    hd = [torch.from_numpy(h).to(dev) for h in heads]
    plug = P.YoloLayerPluginV3()
    out = torch.zeros((B, plug.output_elems()), dtype=torch.float32, device=dev)
    assert plug.enqueue(hd, [out]) == 0
    got = out.cpu().numpy()
    orc, orc_idx = oracle.yolov3_decode(heads, V3_ANCHORS)
    assert np.array_equal(gold[f"v3_{net[0]}_{B}_counts"], got[:, 0]) and np.array_equal(orc[:, 0], got[:, 0]) and got[:, 0].min() > 50
    n_class_gated = 0
    for b in range(B):
        r, g = gold[f"v3_{net[0]}_{B}_{b}"], _canon(_rows(got, b, 7))
        assert oracle.digest(g[:, 4:]) == gold[f"v3_{net[0]}_{B}_{b}_conf"]    # both confidences and the class: bit-exact
        g = g[oracle.sample_index(len(g))]   # the rows stored in r
        np.testing.assert_allclose(g[:, :4], r[:, :4], rtol=3e-7, atol=0)  # same expf; FMA contraction of the reference build
        np.testing.assert_allclose(_rows(got, b, 7), _rows(orc, b, 7), atol=ATOL, rtol=2e-6)
        n_class_gated += int((_rows(got, b, 7)[:, 6] < 0.5).sum())
    assert n_class_gated > 0
    # fused decode + NMS == oracle nms() of yolov3-spp.cpp:77-120 (cxcywh IoU, det_confidence order): variant 1 on 7-float rows
    fused = P.FusedYoloDecodeNms(plug, B, 0.5, 0.4, device=dev)
    comp, idx = fused.enqueue(B, hd)
    comp, idx = comp.cpu().numpy(), idx.cpu().numpy()
    for b in range(B):
        res, src = oracle.nms(1, orc[b], 1000, 7, 0.5, 0.4)
        n = int(comp[b, 0])
        assert n == len(res) and n > 5
        assert np.array_equal(idx[b, :n], orc_idx[b][src])
        np.testing.assert_allclose(comp[b, 1:1 + n * 7].reshape(n, 7)[:, :6], res[:, :6], atol=ATOL, rtol=2e-6)
    q = P.YoloLayerPluginV3.deserialize(plug.serialize())
    assert q.serialize() == plug.serialize() and len(plug.serialize()) == plug.getSerializationSize()


# ------------------------------------------------------------------ yolo26 gather -------------------------
@pytest.mark.parametrize("obb", [False, True])
def test_yolo26_gather_vs_reference_kernel_and_oracle(oracle, dev, gold, obb):
    nc, A, K, B = (15, 21504, 300, 3) if obb else (80, 8400, 300, 3)
    rows = synth.yolo26_rows(B, seed=630 + int(obb), nc=nc, anchors=A, obb=obb)
    rd = torch.from_numpy(rows).to(dev)
    plug = P.YoloLayerPlugin26(nc, 17, K, not obb, False, False, obb, A, conf_thresh=0.3)
    out = torch.full((B, plug.output_elems()), 7.0, dtype=torch.float32, device=dev)
    ws = torch.empty(plug.getWorkspaceSize(B), dtype=torch.uint8, device=dev)
    assert plug.enqueue(B, [rd], [out], ws) == 0
    got = out.cpu().numpy()
    orc, orc_idx = oracle.yolo26_gather(rows, nc=nc, obb=obb, max_out=K, conf_thresh=0.3)
    assert np.array_equal(got, orc)          # pure gather: every float of the buffer, ascending anchor order, zeros elsewhere
    assert 30 < got[:, 0].min() <= got[:, 0].max() <= K
    # the reference decodes image 0 of the batch only (yololayer.cu:185): it ran one image at a time (and zeroed its buffer
    # past the rows, as ours is)
    for b in range(B):
        assert gold[f"v26_{obb}_{b}_count"] == got[b, 0]
        assert oracle.digest(_canon(_rows(got, b, 90))) == gold[f"v26_{obb}_{b}"]
        assert np.all(got[b, 1 + int(got[b, 0]) * 90:] == 0)
    q = P.YoloLayerPlugin26.deserialize(plug.serialize())
    assert q.serialize() == plug.serialize() and len(plug.serialize()) == 24


def test_yolo26_gather_overflow_unaligned_and_empty(oracle, dev):
    # more candidates than max_detections (count clamped, first K in anchor order), a channel count that is not a multiple of
    # 4 (scalar load path), an anchor count that is not a multiple of 32, and an image without candidates
    nc, A, K, B = 3, 1000 + 13, 50, 2
    rows = synth.yolo26_rows(B, seed=640, nc=nc, anchors=A, n_obj=200)
    rows[1, :, 4:] = 0.01
    plug = P.YoloLayerPlugin26(nc, 17, K, True, False, False, False, A, conf_thresh=0.3)
    out = torch.zeros((B, plug.output_elems()), dtype=torch.float32, device=dev)
    ws = torch.empty(plug.getWorkspaceSize(B), dtype=torch.uint8, device=dev)
    assert plug.enqueue(B, [torch.from_numpy(rows).to(dev)], [out], ws) == 0
    got = out.cpu().numpy()
    orc, _ = oracle.yolo26_gather(rows, nc=nc, max_out=K, conf_thresh=0.3)
    assert orc[0, 0] > K and got[0, 0] == K and got[1, 0] == 0
    assert np.array_equal(got[:, 1:], orc[:, 1:])


# ------------------------------------------------------------------ retinafaceAntiCov ---------------------
def test_anticov_decode_vs_reference_kernel_and_oracle(oracle, dev, gold):
    B = 3
    heads = synth.anticov_heads(B, seed=650)
    hd = [torch.from_numpy(h).to(dev) for h in heads]
    plug = P.DecodePlugin(640, 640, anticov=True)
    out = torch.zeros((B, plug.output_elems()), dtype=torch.float32, device=dev)
    ws = torch.empty(plug.getWorkspaceSize(B), dtype=torch.uint8, device=dev)
    assert plug.enqueue(B, hd, [out], ws) == 0
    got = out.cpu().numpy()
    orc, _ = oracle.anticov_decode(heads)
    assert np.array_equal(got[:, 0], orc[:, 0]) and got[:, 0].min() > 50
    for b in range(B):
        np.testing.assert_allclose(_rows(got, b, 16), _rows(orc, b, 16), atol=ATOL, rtol=2e-6)
        # the reference is batch 1 only (no image offset): it ran image by image
        assert gold[f"anticov_{b}_count"] == got[b, 0]
        assert oracle.digest(_canon(_rows(got, b, 16))) == gold[f"anticov_{b}"]   # same expf, same contraction: bit-exact
    # NMS of retinafaceAntiCov.cpp:92-127 = the retinaface host nms() on 16-float rows (landmarks + mask conf ride along)
    comp, idx = P.batch_nms(out, B, plug.output_elems(), P.float_le_threshold(0.1), 0.4, det_floats=16, box_format=L.BOX_RETINA,
                            extra_floats=11, extra_offset=5, max_det=1000, return_index=True)
    comp, idx = comp.cpu().numpy(), idx.cpu().numpy()
    for b in range(B):
        res, src = oracle.nms(2, got[b], plug.total_priors, 16, 0.1, 0.4)
        n = int(comp[b, 0])
        assert n == len(res) and np.array_equal(idx[b, :n], src)
        rows = comp[b, 1:1 + n * 18].reshape(n, 18)
        assert np.array_equal(rows[:, :5], res[:, :5]) and np.array_equal(rows[:, 7:], res[:, 5:])
