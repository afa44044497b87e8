"""Parity against the REFERENCE'S OWN CUDA KERNELS on a B200: the reference's plugin / helper sources, compiled by
oracle/Makefile against the mock NvInfer.h and the OpenCV shim, were run on the inputs below through their public entry
points (plugin enqueue(), free functions), and what they returned is stored in tests/golden/ref_kernels.npz
(tools/make_golden_vs_ref.py device).  These are the strongest parity checks of the suite: same inputs, the reference's
code vs ours.  Outputs compared bit for bit are stored as oracle.digest() strings, the others as arrays.
The reference's slot order is atomicAdd arrival, so decode outputs are compared as canonically sorted sets."""
from pathlib import Path

import numpy as np
import pytest
import torch

from tensorrtx_b200 import _lib as L
from tensorrtx_b200 import plugins as P
from tensorrtx_b200 import synth

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).resolve().parent / "golden" / "ref_kernels.npz"


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _canon(rows):
    order = np.lexsort(tuple(rows[:, k] for k in range(rows.shape[1] - 1, -1, -1)))
    return rows[order]


def _ours_decode(plug, hd, B, dev):
    out = torch.zeros((B, plug.output_elems()), dtype=torch.float32, device=dev)
    ws = torch.empty(plug.getWorkspaceSize(B), dtype=torch.uint8, device=dev)
    assert plug.enqueue(B, hd, [out], ws) == 0
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("seed,B", [(0, 1), (1, 8)])
def test_yolov8_plugin_vs_reference_kernel(dev, oracle, gold, seed, B):
    heads = synth.yolov8_heads(B, seed=400 + seed)
    hd = [torch.from_numpy(h).to(dev) for h in heads]
    counts = gold[f"v8_{seed}_{B}_counts"]
    got = _ours_decode(P.YoloLayerPlugin(80, 17, 0.0, 640, 640, 1000, False, False, False, (8, 16, 32)), hd, B, dev)
    assert np.array_equal(counts, got[:, 0]) and counts.min() > 100
    for b in range(B):
        n = int(counts[b])
        g = _canon(got[b, 1:1 + n * 90].reshape(n, 90)[:, :6])
        assert oracle.digest(g) == gold[f"v8_{seed}_{B}_{b}"]  # same CUDA expf, same operation order: bit-exact


def test_yolov8_near_ulp_sigmoid_collisions_vs_reference_kernel(dev, oracle, gold):
    """Logits a few ulps apart: whether two of them round to the same probability (-> the EARLIER class wins the
    reference's strict `p > max`) depends on expf itself, so this is checked against the reference kernel (same CUDA
    expf), for every scan variant (class slices merge their running state; the TMA pipeline replays from smem)."""
    heads = synth.yolov8_heads(1, seed=430, n_obj=0)
    h = heads[0]
    n = 0
    for x0 in (0.3, 1.5, 2.75, 5.0, 9.0, 14.0):
        x = np.float32(x0)
        for k in range(1, 25):
            y = x
            for _ in range(k):
                y = np.nextafter(y, np.float32(0))
            cell = 40 * n + k
            h[0, 4 + 60 - k, cell] = y      # earlier class, k ulps below the maximum
            h[0, 4 + 60, cell] = x
            h[0, 4 + 70, cell] = y          # later class: never wins
        n += 1
    hd = [torch.from_numpy(a).to(dev) for a in heads]
    nref = int(gold["v8_ulp_count"][0])
    assert nref >= 6 * 24
    plug = P.YoloLayerPlugin(80, 17, 0.0, 640, 640, 1000, False, False, False, (8, 16, 32))
    for pipe, slices, unroll in ((1, 2, 5), (0, 2, 5), (0, 4, 10), (0, 1, 8), (0, 8, 5)):
        plug.tune(tma=pipe, slices=slices, rows=unroll)
        got = _ours_decode(plug, hd, 1, dev)
        assert got[0, 0] == nref
        g = _canon(got[0, 1:1 + nref * 90].reshape(nref, 90)[:, :6])
        assert (g[:, 5] == 60).any() and (g[:, 5] != 60).any()     # both outcomes occur
        assert oracle.digest(g) == gold["v8_ulp"], (pipe, slices, unroll)


@pytest.mark.parametrize("mode", ["seg", "pose", "obb"])
def test_yolov8_plugin_extras_vs_reference_kernel(dev, oracle, gold, mode):
    seg, pose, obb = mode == "seg", mode == "pose", mode == "obb"
    nc = 1 if pose else (15 if obb else 80)
    extra = 32 if seg else (51 if pose else 1)
    B = 2
    heads = synth.yolov8_heads(B, seed=410, nc=nc, extra=extra, n_obj=20)
    hd = [torch.from_numpy(h).to(dev) for h in heads]
    got = _ours_decode(P.YoloLayerPlugin(nc, 17, 0.3, 640, 640, 1000, seg, pose, obb, (8, 16, 32)), hd, B, dev)
    assert np.array_equal(gold[f"v8_{mode}_counts"], got[:, 0])
    cols = list(range(6)) + (list(range(6, 38)) if seg else []) + (list(range(38, 89)) if pose else []) + ([89] if obb else [])
    for b in range(B):
        n = int(got[b, 0])
        r = gold[f"v8_{mode}_{b}"]   # the oracle.sample_index() rows of the reference's canonically sorted rows
        g = _canon(got[b, 1:1 + n * 90].reshape(n, 90)[:, cols])[oracle.sample_index(n)]
        np.testing.assert_allclose(g, r, rtol=1e-6, atol=1e-6)  # obb/pose use fp64 sin/cos/mul in both


def test_yolov5_plugin_vs_reference_kernel(dev, oracle, gold):
    B = 4
    heads = synth.yolov5_heads(B, seed=420)
    hd = [torch.from_numpy(h).to(dev) for h in heads]
    kern = [P.YoloKernel(640 // s, 640 // s, a) for s, a in zip((8, 16, 32), synth.V5_ANCHORS)]
    got = _ours_decode(P.YoloLayerPluginV5(80, 640, 640, 1000, False, kern), hd, B, dev)
    counts = gold["v5_counts"]
    assert np.array_equal(counts, got[:, 0]) and counts.min() > 100
    for b in range(B):
        n = int(counts[b])
        r = gold[f"v5_{b}"]   # the oracle.sample_index() rows of the reference's canonically sorted rows
        g = _canon(got[b, 1:1 + n * 38].reshape(n, 38)[:, :6])[oracle.sample_index(n)]
        np.testing.assert_allclose(g, r, rtol=3e-7, atol=0)  # FMA contraction of the reference build: <= 2 ulp


def test_retina_plugin_vs_reference_kernel(dev, oracle, gold):
    h, w = 480, 640   # the input size the reference's retinaface/decode.h compiles in
    B = 4
    heads = synth.retina_heads(B, seed=430, in_h=h, in_w=w)
    hd = [torch.from_numpy(x).to(dev) for x in heads]
    plug = P.DecodePlugin(h, w)
    out = torch.zeros((B, plug.output_elems()), dtype=torch.float32, device=dev)
    assert plug.enqueue(B, hd, [out], torch.empty(plug.getWorkspaceSize(B), dtype=torch.uint8, device=dev)) == 0
    got = out.cpu().numpy()
    counts = gold["retina_counts"]
    assert np.array_equal(counts, got[:, 0]) and counts.min() > 50
    for b in range(B):
        n = int(counts[b])
        r = gold[f"retina_{b}"]   # the oracle.sample_index() rows of the reference's canonically sorted rows
        g = _canon(got[b, 1:1 + n * 15].reshape(n, 15))[oracle.sample_index(n)]
        np.testing.assert_allclose(g, r, rtol=3e-7, atol=1e-5)


def test_cuda_decode_nms_vs_reference_kernels(dev, oracle, gold):
    heads = synth.yolov8_heads(1, seed=440)
    plugin_out, _ = oracle.yolov8_decode(heads)
    pd = torch.from_numpy(plugin_out).to(dev)
    comp = P.batch_nms(pd, 1, plugin_out.shape[1], 0.5, 0.45, mode=L.NMS_ONESHOT).cpu().numpy()
    n = int(comp[0, 0])
    gg = comp[0, 1:1 + n * 7].reshape(n, 7)
    assert n == gold["cuda_decode_nms_n"]                 # the reference's rows above conf (holes stay zero there)
    assert oracle.digest(_canon(gg)) == gold["cuda_decode_nms"]   # identical rows AND identical keep flags


def test_preprocess_vs_reference_kernel(dev, oracle, gold):
    # 640x640 / 640x480 / 480x640 / 416x640: scale == 1 -> the TMA-staged unit-scale kernel (incl. padding and border
    # tiles); 500x640 has a pitch TMA cannot take (1500 B) -> general kernel at scale 1; the others resample.
    for (h, w) in [(640, 640), (1080, 1920), (375, 500), (480, 640), (640, 480), (416, 640), (640, 500), (639, 640), (640, 624)]:
        img = synth.frames(1, seed=h, h=h, w=w)[0]
        dst = torch.zeros((1, 3, 640, 640), dtype=torch.float32, device=dev)
        P.cuda_batch_preprocess([torch.from_numpy(img).to(dev)], dst, 640, 640)
        torch.cuda.synchronize()
        # both builds leave the bilinear sum to nvcc's FMA contraction: bit-identical
        assert oracle.digest(dst[0].cpu().numpy()) == gold[f"preprocess_{h}x{w}"], (h, w)


def test_rcnn_vs_reference_functions(dev, oracle, gold):
    B, A, H, W, top_n = 2, 15, 50, 67, 6000
    scores, deltas = synth.rpn_inputs(B, seed=450, A=A, H=H, W=W)
    anchors = synth.rcnn_anchors()
    sd, dd = torch.from_numpy(scores).to(dev), torch.from_numpy(deltas).to(dev)
    plug = P.RpnDecodePlugin(top_n, anchors, 16.0, 800, 1067, H, W)
    os_, ob = torch.zeros((B, top_n), device=dev), torch.zeros((B, top_n, 4), device=dev)
    ws = torch.empty(256, dtype=torch.uint8, device=dev)
    assert plug.enqueue(B, [sd, dd], [os_, ob], ws) == 0
    assert oracle.digest(os_.cpu().numpy()) == gold["rpn_scores"]          # same ordered top-6000
    # the reference's boxes: the first `pre` rows (the RpnNms input below) and a fixed sample of the others
    pre, post = 1000, 300
    rb_pre, rows = gold["rpn_boxes_pre"], gold["rpn_boxes_rows"]
    np.testing.assert_allclose(ob[:, :pre].cpu().numpy(), rb_pre, rtol=3e-7, atol=1e-4)
    np.testing.assert_allclose(ob[:, rows].cpu().numpy(), gold["rpn_boxes_sample"], rtol=3e-7, atol=1e-4)

    # RpnNms on <= 1024 boxes (the reference kernel is only race-free within one block; it ran once per image, being only
    # correct for batch 1: its second sort overwrites the iota `indices` buffer that the next image's first sort uses as
    # payload, RpnNms.cu:100 vs :112-113), on the reference's scores and boxes
    s1, b1 = os_[:, :pre].contiguous(), torch.from_numpy(rb_pre).to(dev)
    onb = torch.zeros((B, post, 4), device=dev)
    assert P.RpnNmsPlugin(0.7, post, pre).enqueue(B, [s1, b1], [onb], ws) == 0
    orc = oracle.rpn_nms(s1.cpu().numpy(), rb_pre, post, 0.7)
    assert oracle.digest(onb.cpu().numpy()) == gold["rpn_nms"], \
        f"rows differing from the oracle: ours {int((onb.cpu().numpy() != orc).any(-1).sum())}"



def test_rcnn_predictor_and_batched_nms_vs_reference_functions(dev, oracle, gold):
    B = 2
    ws = torch.empty(256, dtype=torch.uint8, device=dev)
    # PredictorDecode + BatchedNms (count = 1000: one block)
    N, Cc = 1000, 80
    sc, dl, pr = synth.predictor_inputs(B, seed=451, N=N, Ccls=Cc)
    scd, dld, prd = (torch.from_numpy(x).to(dev) for x in (sc, dl, pr))
    o1, o2, o3 = (torch.zeros((B, N), device=dev), torch.zeros((B, N, 4), device=dev), torch.zeros((B, N), device=dev))
    assert P.PredictorDecodePlugin(N, 800, 1067, (10.0, 10.0, 5.0, 5.0), Cc).enqueue(B, [scd, dld, prd], [o1, o2, o3], ws) == 0
    assert oracle.digest(o1.cpu().numpy()) == gold["pred_scores"] and oracle.digest(o3.cpu().numpy()) == gold["pred_classes"]
    r2 = gold["pred_boxes"]
    np.testing.assert_allclose(o2.cpu().numpy(), r2, rtol=3e-7, atol=1e-4)
    # BatchedNms on the reference's outputs (scores and classes are ours: identical above); the reference ran once per
    # image (same batch > 1 bug as RpnNms, BatchedNms.cu:134 vs :146-148)
    r1, r2d, r3 = o1, torch.from_numpy(r2).to(dev), o3
    for method in (0, 1, 2):
        q1 = gold[f"bnms_{method}_scores"]
        p1, p2, p3 = torch.zeros((B, 100), device=dev), torch.zeros((B, 100, 4), device=dev), torch.zeros((B, 100), device=dev)
        assert P.BatchedNmsPlugin(method, 0.5, 100, N).enqueue(B, [r1, r2d, r3], [p1, p2, p3], ws) == 0
        _, ob_, _ = oracle.batched_nms(method, r1.cpu().numpy(), r2, r3.cpu().numpy(), 100, 0.5)
        info = f"method {method}: rows differing from the oracle: ours {int((p2.cpu().numpy() != ob_).any(-1).sum())}"
        np.testing.assert_allclose(p1.cpu().numpy(), q1, rtol=1e-6, atol=0, err_msg=info)
        assert oracle.digest(p2.cpu().numpy()) == gold[f"bnms_{method}_boxes"], info
        assert oracle.digest(p3.cpu().numpy()) == gold[f"bnms_{method}_classes"], info


def test_roi_align_and_mask_rcnn_inference_vs_reference_functions(dev, oracle, gold):
    """roiAlign / maskRcnnInference of rcnn/*.cu (one launch + cudaDeviceSynchronize per image there) vs one launch
    for the batch here: same CUDA compiler, same expressions -> identical floats."""
    rng = np.random.default_rng(470)
    B, N, Cc, H, W, Pp = 2, 96, 80, 50, 67, 14
    feat = rng.standard_normal((B, Cc, H, W)).astype(np.float32)
    x1 = rng.uniform(-40, 1000, (B, N)); y1 = rng.uniform(-40, 760, (B, N))
    w = np.exp(rng.uniform(np.log(8), np.log(900), (B, N))); h = np.exp(rng.uniform(np.log(8), np.log(700), (B, N)))
    rois = np.stack([x1, y1, x1 + w, y1 + h], -1).astype(np.float32)
    rois[0, 0] = [100, 100, 100, 100]        # zero-size proposal: count = 0 -> NaN, like the reference
    rois[0, 1] = [300, 300, 200, 250]        # negative size
    rois[1, 0] = [-500, -500, -300, -300]    # entirely outside the feature map
    xi = rng.uniform(0, 700, N); yi = rng.uniform(0, 500, N)
    wi = np.exp(rng.uniform(np.log(8), np.log(300), N)); hi = np.exp(rng.uniform(np.log(8), np.log(250), N))
    rois_in = np.stack([xi, yi, xi + wi, yi + hi], -1).astype(np.float32)
    fd, rd = torch.from_numpy(feat).to(dev), torch.from_numpy(rois).to(dev)
    rois[1, 1] = [0, 0, 1067, 800]           # the whole map: the window of a channel is 50 x 67 cells (several passes)
    rois[1, 2] = [5, 5, 9, 9]                # a fraction of one cell
    rois[1, 3] = [1060, 790, 1200, 900]      # hangs over the bottom-right corner
    for sampling in (0, 2, 5, 19):           # 19: 14 * 19 = 266 table entries per axis > 256 -> coordinates on the fly
        plug = P.RoiAlignPlugin(Pp, 1 / 16, sampling, N, Cc)
        plug.configurePlugin([(N, 4), (Cc, H, W)])
        for mode in (None, L.ROI_WINDOW, L.ROI_DIRECT):  # the shared-memory window kernel (default) and the round-1 kernel
            got = torch.full((B, N, Cc, Pp, Pp), -3.0, device=dev)
            assert plug.enqueue(B, [rd, fd], [got], mode=mode) == 0
            torch.cuda.synchronize()
            g = got.cpu().numpy()
            # NaN where the reference has NaN, its bits everywhere else
            assert oracle.digest(np.stack([np.isnan(g), np.nan_to_num(g, nan=0.0)]).astype(np.float32)) == \
                gold[f"roi_align_{sampling}"], (sampling, mode)
        if sampling > 2:
            continue
        # CPU restatement (no FMA contraction) on proposals inside the feature map: at the `x > width -> 0` border of
        # bilinear_interpolate a 1-ulp difference in a sample coordinate flips a whole tap, which only the same-compiler
        # comparison above can pin
        orc = oracle.roi_align(rois_in, feat[1], Pp, 1 / 16, sampling)
        got_in = torch.empty((1, N, Cc, Pp, Pp), device=dev)
        assert plug.enqueue(1, [torch.from_numpy(rois_in).to(dev), fd[1:2].contiguous()], [got_in]) == 0
        np.testing.assert_allclose(got_in[0].cpu().numpy(), orc, rtol=0, atol=2e-5)
    # MaskRcnnInference
    D, nc, S = 100, 80, 14
    masks = rng.standard_normal((B, D, nc, S, S)).astype(np.float32) * 3
    idx = rng.integers(0, nc, (B, D)).astype(np.float32)
    idx[0, 5] = -1.0
    idx[1, 7] = float(nc)                      # out of range: the row is not written
    md, idd = torch.from_numpy(masks).to(dev), torch.from_numpy(idx).to(dev)
    got = torch.full((B, D, S, S), 9.0, device=dev)
    assert P.MaskRcnnInferencePlugin(D, S, nc).enqueue(B, [idd, md], [got]) == 0
    torch.cuda.synchronize()
    assert oracle.digest(got.cpu().numpy()) == gold["mask_rcnn_inference"]
    assert torch.all(got[0, 5] == 9.0) and torch.all(got[1, 7] == 9.0)
    exp = oracle.mask_rcnn_inference(idx[1], masks[1], out=np.full((D, S, S), 9.0, np.float32))
    np.testing.assert_allclose(got[1].cpu().numpy(), exp, rtol=3e-7, atol=1e-7)

