"""Golden data of the reference's own compiled code for the parity tests that used to call it directly:

    python tools/make_golden_vs_ref.py host           -> tests/golden/oracle_vs_ref.npz  (tests/test_oracle_vs_ref_cpu.py)
    python tools/make_golden_vs_ref.py device DIR     -> DIR/ref_kernels.npz             (tests/test_vs_reference_gpu.py,
                                                                                           tests/test_variants_gpu.py)

Needs oracle/_ref/, which `make -C oracle` compiles from a checkout of the reference (REF=...); `device` also needs a B200.
Every input is rebuilt from the same seeds as in the tests.  Outputs the tests compare bit for bit are stored as
oracle.digest() strings, outputs they compare with a tolerance (or feed to a later stage) as arrays; of decode rows, the
oracle.sample_index() rows of each image."""
import ctypes as C
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from oracle import oracle as O  # noqa: E402
from tensorrtx_b200 import synth  # noqa: E402

REF = ROOT / "oracle" / "_ref"
D = O.digest


def _lib(name):
    return C.CDLL(str(REF / name))


def _ref_nms(fn, buf, F, *thr):
    out = np.zeros((buf.shape[0] // F + 1) * F, np.float32)
    b = np.ascontiguousarray(buf, np.float32)
    n = fn(b.ctypes.data_as(C.c_void_p), *[C.c_float(t) for t in thr], out.ctypes.data_as(C.c_void_p))
    return out[:n * F].reshape(n, F).copy()


SIZES = ((1920, 1080), (1080, 1920), (640, 640), (1280, 720), (333, 777), (4000, 3000), (641, 640), (50, 60))


def host() -> dict:
    v8, v5, rt = _lib("libref_yolov8_host.so"), _lib("libref_yolov5_host.so"), _lib("libref_retina_host.so")
    g = {}

    def nms(key, ref):
        g[key + "_n"], g[key] = np.int32(len(ref)), D(ref)

    for seed in range(4):
        out, _ = O.yolov8_decode(synth.yolov8_heads(2, seed=100 + seed))
        for b in range(2):
            nms(f"v8_nms_{seed}_{b}", _ref_nms(v8.ref_v8_nms, out[b], 90, 0.5, 0.45))
    for seed in range(3):
        out, _ = O.yolov8_decode(synth.yolov8_heads(2, seed=130 + seed, nc=15, extra=1, n_obj=40), nc=15, is_obb=True)
        for b in range(2):
            for thr in (0.5, 0.2):
                nms(f"v8_obb_{seed}_{b}_{thr}", _ref_nms(v8.ref_v8_nms_obb, out[b], 90, 0.3, thr))
    rng = np.random.default_rng(1)
    n = 400
    buf = np.zeros(1 + 1000 * 90, np.float32)
    rows = buf[1:1 + n * 90].reshape(n, 90)
    xy = rng.uniform(0, 600, (n, 2))
    wh = rng.uniform(10, 60, (n, 2))
    rows[:, :2], rows[:, 2:4] = xy, xy + wh
    rows[:, 4] = np.round(rng.uniform(0.5, 1.0, n), 2)
    rows[:, 5] = rng.integers(0, 3, n)
    buf[0] = n
    nms("v8_ties", _ref_nms(v8.ref_v8_nms, buf, 90, 0.5, 0.45))
    out, _ = O.yolov8_decode(synth.yolov8_heads(3, seed=7))
    res = np.zeros((3, 1000, 90), np.float32)
    cnt = np.zeros(3, np.int32)
    v8.ref_v8_batch_nms(np.ascontiguousarray(out).ctypes.data_as(C.c_void_p), 3, out.shape[1], C.c_float(0.3), C.c_float(0.6),
                        res.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p), 1000)
    for b in range(3):
        nms(f"v8_batch_{b}", res[b, :cnt[b]])
    for seed in range(3):
        out, _ = O.yolov5_decode(synth.yolov5_heads(1, seed=200 + seed, n_obj=200), synth.V5_ANCHORS)
        nms(f"v5_nms_{seed}", _ref_nms(v5.ref_v5_nms, out[0], 38, 0.5, 0.45))
    for seed in range(3):
        out, _ = O.retina_decode(synth.retina_heads(1, seed=300 + seed, in_h=480, in_w=640, n_obj=60), in_h=480, in_w=640)
        nms(f"retina_nms_{seed}", _ref_nms(rt.ref_retina_nms, out[0], 15, 0.4))
    tp = O.retina_total_priors(480, 640)
    buf = np.zeros(1 + tp * 15, np.float32)
    buf[0] = 3
    for i, c in enumerate([np.float32(0.1), np.nextafter(np.float32(0.1), np.float32(0)), np.float32(0.5)]):
        buf[1 + i * 15:1 + i * 15 + 4] = [100 * i, 0, 100 * i + 50, 50]
        buf[1 + i * 15 + 4] = c
    nms("retina_conf", _ref_nms(rt.ref_retina_nms, buf, 15, 0.4))
    # get_rect: 4000 boxes per variant, the rectangles in test order
    for variant, lib, fn in ((0, v8, "ref_v8_get_rect"), (1, v5, "ref_v5_get_rect")):
        rng = np.random.default_rng(50 + variant)
        rects = []
        for (w, h) in SIZES:
            for _ in range(500):
                if variant == 0:
                    x1, y1 = rng.uniform(-30, 650, 2)
                    bb = np.array([x1, y1, x1 + rng.uniform(-5, 400), y1 + rng.uniform(-5, 400)], np.float32)
                else:
                    bb = np.array([rng.uniform(-30, 670), rng.uniform(-30, 670), rng.uniform(0, 500), rng.uniform(0, 500)], np.float32)
                r = np.zeros(4, np.int32)
                getattr(lib, fn)(w, h, bb.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p))
                rects.append(r)
        g[fn] = D(np.array(rects))
    rng = np.random.default_rng(70)
    rects, lmks = [], []
    for (w, h) in SIZES:
        for _ in range(300):
            x1, y1 = rng.uniform(-30, 650, 2)
            bb = np.array([x1, y1, x1 + rng.uniform(-5, 400), y1 + rng.uniform(-5, 400)], np.float32)
            lmk = rng.uniform(-20, 660, 51).astype(np.float32)
            lmk[2::3] = rng.uniform(0, 1, 17).astype(np.float32)
            r = np.zeros(4, np.int32)
            v8.ref_v8_get_rect_adapt_landmark(w, h, bb.copy().ctypes.data_as(C.c_void_p), lmk.ctypes.data_as(C.c_void_p),
                                              r.ctypes.data_as(C.c_void_p))
            rects.append(r), lmks.append(lmk)
    g["v8_lmk_rects"], g["v8_lmk"] = D(np.array(rects)), D(np.array(lmks))
    r6s = []
    for w in list(range(37, 2000, 97)) + [640, 641, 1920, 1080]:
        for h in (48, 479, 480, 640, 1080, 1920, 3000):
            r6 = np.zeros(6, np.int32)
            v8.ref_v8_scale_mask_rect(w, h, r6.ctypes.data_as(C.c_void_p))
            r6s.append(r6)
    g["scale_mask_rect"] = np.array(r6s)
    rng = np.random.default_rng(71)
    K = 200
    buf = np.zeros(1 + K * 7, np.float32)
    buf[0] = K
    rows = buf[1:].reshape(K, 7)
    rows[:, :6] = rng.uniform(0, 640, (K, 6)).astype(np.float32)
    rows[:, 6] = rng.integers(0, 2, K)
    out = np.zeros((K, 6), np.float32)
    n = v8.ref_v8_process_decode_ptr_host(buf.ctypes.data_as(C.c_void_p), 7, K, out.ctypes.data_as(C.c_void_p))
    g["pdh"] = out[:n].copy()
    rng = np.random.default_rng(72)
    for elem in (8, 9):
        K = 150
        buf = np.zeros(1 + K * elem, np.float32)
        buf[0] = K
        rows = buf[1:].reshape(K, elem)
        rows[:, :] = rng.uniform(-3, 640, (K, elem)).astype(np.float32)
        rows[:, 6] = rng.integers(0, 3, K)
        out = np.zeros((K, 7), np.float32)
        n = v8.ref_v8_process_decode_ptr_host_obb(buf.ctypes.data_as(C.c_void_p), elem, K, out.ctypes.data_as(C.c_void_p))
        g[f"pdh_obb_{elem}"] = out[:n].copy()
    rng = np.random.default_rng(73)
    rects, lmks = [], []
    for (in_w, in_h) in ((640, 640), (640, 480)):
        for (w, h) in SIZES:
            for _ in range(250):
                x1, y1 = rng.uniform(-30, in_w + 10), rng.uniform(-30, in_h + 10)
                bb = np.array([x1, y1, x1 + rng.uniform(-5, 400), y1 + rng.uniform(-5, 400)], np.float32)
                lmk = rng.uniform(-20, 660, 10).astype(np.float32)
                r = np.zeros(4, np.int32)
                rt.ref_retina_get_rect_adapt_landmark(w, h, in_w, in_h, bb.copy().ctypes.data_as(C.c_void_p), lmk.ctypes.data_as(C.c_void_p),
                                                      r.ctypes.data_as(C.c_void_p))
                rects.append(r), lmks.append(lmk)
    g["retina_lmk_rects"], g["retina_lmk"] = D(np.array(rects)), D(np.array(lmks))
    return g


def canon(rows):
    """rows sorted lexicographically on every column: the reference's slot order is atomicAdd arrival"""
    return rows[np.lexsort(tuple(rows[:, k] for k in range(rows.shape[1] - 1, -1, -1)))]


def _rows(buf, b, F):
    n = int(buf[b, 0])
    return buf[b, 1:1 + n * F].reshape(n, F)


def _sample(rows):
    return rows[O.sample_index(len(rows))]


def device() -> dict:
    import torch

    from tensorrtx_b200 import plugins as P
    dev = torch.device("cuda", 0)
    g = {}

    def ptrs(ts):
        return (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])

    def vp(t):
        return C.c_void_p(t.data_ptr())

    v8 = _lib("libref_yolov8.so")
    strides = (C.c_int * 3)(8, 16, 32)

    def v8_plugin(heads, nc=80, gate=0.0, seg=0, pose=0, obb=0):
        B = heads[0].shape[0]
        hd = [torch.from_numpy(h).to(dev) for h in heads]
        ref = torch.zeros((B, 1 + 1000 * 90), dtype=torch.float32, device=dev)
        assert v8.ref_v8_plugin_enqueue(nc, 17, C.c_float(gate), 640, 640, 1000, seg, pose, obb, strides, 3, B, ptrs(hd), vp(ref), None) == 0
        return ref.cpu().numpy()

    # ---- tests/test_vs_reference_gpu.py ----
    for seed, B in ((0, 1), (1, 8)):
        ref = v8_plugin(synth.yolov8_heads(B, seed=400 + seed))
        g[f"v8_{seed}_{B}_counts"] = ref[:, 0].copy()
        for b in range(B):
            g[f"v8_{seed}_{B}_{b}"] = D(canon(_rows(ref, b, 90)[:, :6]))
    heads = synth.yolov8_heads(1, seed=430, n_obj=0)
    h = heads[0]
    for n, x0 in enumerate((0.3, 1.5, 2.75, 5.0, 9.0, 14.0)):
        x = np.float32(x0)
        for k in range(1, 25):
            y = x
            for _ in range(k):
                y = np.nextafter(y, np.float32(0))
            cell = 40 * n + k
            h[0, 4 + 60 - k, cell], h[0, 4 + 60, cell], h[0, 4 + 70, cell] = y, x, y
    ref = v8_plugin(heads)
    g["v8_ulp_count"], g["v8_ulp"] = ref[:, 0].copy(), D(canon(_rows(ref, 0, 90)[:, :6]))
    for mode in ("seg", "pose", "obb"):
        seg, pose, obb = mode == "seg", mode == "pose", mode == "obb"
        nc = 1 if pose else (15 if obb else 80)
        extra = 32 if seg else (51 if pose else 1)
        ref = v8_plugin(synth.yolov8_heads(2, seed=410, nc=nc, extra=extra, n_obj=20), nc, 0.3, int(seg), int(pose), int(obb))
        cols = list(range(6)) + (list(range(6, 38)) if seg else []) + (list(range(38, 89)) if pose else []) + ([89] if obb else [])
        g[f"v8_{mode}_counts"] = ref[:, 0].copy()
        for b in range(2):
            g[f"v8_{mode}_{b}"] = _sample(canon(_rows(ref, b, 90)[:, cols]))
    v5 = _lib("libref_yolov5.so")
    B = 4
    hd = [torch.from_numpy(h).to(dev) for h in synth.yolov5_heads(B, seed=420)]
    ks = np.zeros((3, 8), np.float32)
    ki = ks.view(np.int32)
    for lvl, (s, a) in enumerate(zip((8, 16, 32), synth.V5_ANCHORS)):
        ki[lvl, 0], ki[lvl, 1] = 640 // s, 640 // s
        ks[lvl, 2:] = a
    ref = torch.zeros((B, 1 + 1000 * 38), dtype=torch.float32, device=dev)
    assert v5.ref_v5_plugin_enqueue(80, 640, 640, 1000, 0, ks.ctypes.data_as(C.c_void_p), 3, B, ptrs(hd), vp(ref), None) == 0
    ref = ref.cpu().numpy()
    g["v5_counts"] = ref[:, 0].copy()
    for b in range(B):
        g[f"v5_{b}"] = _sample(canon(_rows(ref, b, 38)[:, :6]))
    rt = _lib("libref_retina.so")
    assert (rt.ref_retina_input_h(), rt.ref_retina_input_w()) == (480, 640)
    hd = [torch.from_numpy(x).to(dev) for x in synth.retina_heads(B, seed=430, in_h=480, in_w=640)]
    ref = torch.zeros((B, P.DecodePlugin(480, 640).output_elems()), dtype=torch.float32, device=dev)
    assert rt.ref_retina_plugin_enqueue(B, ptrs(hd), vp(ref), None) == 0
    ref = ref.cpu().numpy()
    g["retina_counts"] = ref[:, 0].copy()
    for b in range(B):
        g[f"retina_{b}"] = _sample(canon(_rows(ref, b, 15)))
    plugin_out, _ = O.yolov8_decode(synth.yolov8_heads(1, seed=440))
    pd = torch.from_numpy(plugin_out).to(dev)
    parray = torch.zeros(1 + 1000 * 7, dtype=torch.float32, device=dev)
    assert v8.ref_v8_cuda_decode_nms(vp(pd), 1000, C.c_float(0.5), vp(parray), 1000, C.c_float(0.45), None) == 0
    ref = parray.cpu().numpy()
    rr = ref[1:1 + int(ref[0]) * 7].reshape(-1, 7)
    rr = rr[rr[:, 4] > 0]
    g["cuda_decode_nms_n"], g["cuda_decode_nms"] = np.int32(len(rr)), D(canon(rr))
    for (h, w) in [(640, 640), (1080, 1920), (375, 500), (480, 640), (640, 480), (416, 640), (640, 500), (639, 640), (640, 624)]:
        img = synth.frames(1, seed=h, h=h, w=w)[0]
        ref = torch.zeros((3, 640, 640), dtype=torch.float32, device=dev)
        assert v8.ref_v8_preprocess(img.ctypes.data_as(C.c_void_p), w, h, vp(ref), 640, 640, None) == 0
        g[f"preprocess_{h}x{w}"] = D(ref.cpu().numpy())
    rc = _lib("libref_rcnn.so")
    B, A, H, W, top_n = 2, 15, 50, 67, 6000
    scores, deltas = synth.rpn_inputs(B, seed=450, A=A, H=H, W=W)
    anchors = synth.rcnn_anchors()
    sd, dd = torch.from_numpy(scores).to(dev), torch.from_numpy(deltas).to(dev)
    rs, rb = torch.zeros((B, top_n), device=dev), torch.zeros((B, top_n, 4), device=dev)
    assert rc.ref_rpn_decode(B, vp(sd), vp(dd), vp(rs), vp(rb), H, W, 800, 1067, C.c_float(16.0), anchors.ctypes.data_as(C.c_void_p),
                             A, top_n) == 0
    pre, post = 1000, 300
    rbn = rb.cpu().numpy()
    g["rpn_scores"] = D(rs.cpu().numpy())
    g["rpn_boxes_pre"] = rbn[:, :pre].copy()                          # the RpnNms input
    g["rpn_boxes_rows"] = np.sort(np.random.default_rng(0).choice(np.arange(pre, top_n), 1000, replace=False))
    g["rpn_boxes_sample"] = rbn[:, g["rpn_boxes_rows"]].copy()       # a fixed sample of the rest
    s1, b1 = rs[:, :pre].contiguous(), rb[:, :pre].contiguous()
    rnb = torch.zeros((B, post, 4), device=dev)
    for b in range(B):   # batch 1 per call: the reference's second sort clobbers the next image's payload (RpnNms.cu:100 vs :112-113)
        assert rc.ref_rpn_nms(1, vp(s1[b]), vp(b1[b]), vp(rnb[b]), pre, post, C.c_float(0.7)) == 0
    g["rpn_nms"] = D(rnb.cpu().numpy())
    N, Cc = 1000, 80
    sc, dl, pr = synth.predictor_inputs(B, seed=451, N=N, Ccls=Cc)
    scd, dld, prd = (torch.from_numpy(x).to(dev) for x in (sc, dl, pr))
    w4 = (C.c_float * 4)(10.0, 10.0, 5.0, 5.0)
    r1, r2, r3 = torch.zeros((B, N), device=dev), torch.zeros((B, N, 4), device=dev), torch.zeros((B, N), device=dev)
    assert rc.ref_predictor_decode(B, vp(scd), vp(dld), vp(prd), vp(r1), vp(r2), vp(r3), N, Cc, 800, 1067, w4) == 0
    g["pred_scores"], g["pred_boxes"], g["pred_classes"] = D(r1.cpu().numpy()), r2.cpu().numpy(), D(r3.cpu().numpy())
    for method in (0, 1, 2):
        q1, q2, q3 = torch.zeros((B, 100), device=dev), torch.zeros((B, 100, 4), device=dev), torch.zeros((B, 100), device=dev)
        for b in range(B):   # same batch > 1 bug as RpnNms (BatchedNms.cu:134 vs :146-148)
            assert rc.ref_batched_nms(method, 1, vp(r1[b]), vp(r2[b]), vp(r3[b]), vp(q1[b]), vp(q2[b]), vp(q3[b]), N, 100, C.c_float(0.5)) == 0
        g[f"bnms_{method}_scores"], g[f"bnms_{method}_boxes"], g[f"bnms_{method}_classes"] = \
            q1.cpu().numpy(), D(q2.cpu().numpy()), D(q3.cpu().numpy())
    rng = np.random.default_rng(470)
    B, N, Cc, H, W, Pp = 2, 96, 80, 50, 67, 14
    feat = rng.standard_normal((B, Cc, H, W)).astype(np.float32)
    x1 = rng.uniform(-40, 1000, (B, N)); y1 = rng.uniform(-40, 760, (B, N))                                   # noqa: E702
    w = np.exp(rng.uniform(np.log(8), np.log(900), (B, N))); h = np.exp(rng.uniform(np.log(8), np.log(700), (B, N)))  # noqa: E702
    rois = np.stack([x1, y1, x1 + w, y1 + h], -1).astype(np.float32)
    rois[0, 0], rois[0, 1], rois[1, 0] = [100, 100, 100, 100], [300, 300, 200, 250], [-500, -500, -300, -300]
    rng.uniform(0, 700, N); rng.uniform(0, 500, N); rng.uniform(size=N); rng.uniform(size=N)                   # noqa: E702  (rois_in)
    fd, rd = torch.from_numpy(feat).to(dev), torch.from_numpy(rois).to(dev)   # the device copy is taken before the last three edits
    for sampling in (0, 2, 5, 19):
        ref = torch.zeros((B, N, Cc, Pp, Pp), device=dev)
        assert rc.ref_roi_align(B, vp(rd), vp(fd), vp(ref), Pp, C.c_float(1 / 16), sampling, N, Cc, H, W) == 0
        r = ref.cpu().numpy()
        g[f"roi_align_{sampling}"] = D(np.stack([np.isnan(r), np.nan_to_num(r, nan=0.0)]).astype(np.float32))
    D_, nc, S = 100, 80, 14
    masks = rng.standard_normal((B, D_, nc, S, S)).astype(np.float32) * 3
    idx = rng.integers(0, nc, (B, D_)).astype(np.float32)
    idx[0, 5], idx[1, 7] = -1.0, float(nc)
    md, idd = torch.from_numpy(masks).to(dev), torch.from_numpy(idx).to(dev)
    ref = torch.full((B, D_, S, S), 9.0, device=dev)
    assert rc.ref_mask_rcnn_inference(B, vp(idd), vp(md), vp(ref), D_, S, nc) == 0
    g["mask_rcnn_inference"] = D(ref.cpu().numpy())

    # ---- tests/test_variants_gpu.py ----
    v7 = _lib("libref_yolov7.so")
    assert v7.ref_v7_det_floats() == 6
    B = 3
    hd = [torch.from_numpy(h).to(dev) for h in synth.yolov5_heads(B, seed=610)]
    ref = torch.zeros((B, 1 + 1000 * 6), dtype=torch.float32, device=dev)
    assert v7.ref_v7_plugin_enqueue(80, 640, 640, 1000, ks.ctypes.data_as(C.c_void_p), 3, B, ptrs(hd), vp(ref), None) == 0
    ref = ref.cpu().numpy()
    g["v7_counts"] = ref[:, 0].copy()
    for b in range(B):
        g[f"v7_{b}"] = _sample(canon(_rows(ref, b, 6)))
    v3 = _lib("libref_yolov3.so")
    assert v3.ref_v3_det_floats() == 7 and v3.ref_v3_num_classes() == 80
    for net, B in (((608, 608), 2), ((416, 352), 3)):
        heads = synth.yolov3_heads(B, seed=620 + B, net_w=net[0], net_h=net[1])
        hd = [torch.from_numpy(h).to(dev) for h in heads]
        gh, gw = (C.c_int * 3)(*[h.shape[2] for h in heads]), (C.c_int * 3)(*[h.shape[3] for h in heads])
        ref = torch.zeros((B, 1 + 1000 * 7), dtype=torch.float32, device=dev)
        assert v3.ref_v3_plugin_enqueue(B, gh, gw, ptrs(hd), vp(ref)) == 0
        ref = ref.cpu().numpy()
        g[f"v3_{net[0]}_{B}_counts"] = ref[:, 0].copy()
        for b in range(B):
            r = canon(_rows(ref, b, 7))
            g[f"v3_{net[0]}_{B}_{b}"], g[f"v3_{net[0]}_{B}_{b}_conf"] = _sample(r), D(r[:, 4:])
    v26 = _lib("libref_yolo26.so")
    assert v26.ref_v26_det_floats() == 90
    for obb in (False, True):
        nc, A, K, B = (15, 21504, 300, 3) if obb else (80, 8400, 300, 3)
        rd = torch.from_numpy(synth.yolo26_rows(B, seed=630 + int(obb), nc=nc, anchors=A, obb=obb)).to(dev)
        for b in range(B):   # the reference decodes image 0 of a batch only (yololayer.cu:185)
            ref = torch.full((1, 1 + K * 90), 3.0, dtype=torch.float32, device=dev)
            assert v26.ref_v26_plugin_enqueue(nc, 17, K, int(not obb), int(obb), A, C.c_float(0.3), vp(rd[b]), vp(ref), None) == 0
            ref = ref.cpu().numpy()
            assert np.all(ref[0, 1 + int(ref[0, 0]) * 90:] == 0)
            g[f"v26_{obb}_{b}_count"], g[f"v26_{obb}_{b}"] = ref[0, 0], D(canon(_rows(ref, 0, 90)))
    ac = _lib("libref_anticov.so")
    assert (ac.ref_anticov_input_h(), ac.ref_anticov_input_w(), ac.ref_anticov_det_floats()) == (640, 640, 16)
    B = 3
    hd = [torch.from_numpy(h).to(dev) for h in synth.anticov_heads(B, seed=650)]
    for b in range(B):   # batch 1 only (no image offset)
        ref = torch.zeros((1, P.DecodePlugin(640, 640, anticov=True).output_elems()), dtype=torch.float32, device=dev)
        assert ac.ref_anticov_plugin_enqueue(ptrs([x[b:b + 1].contiguous() for x in hd]), vp(ref)) == 0
        ref = ref.cpu().numpy()
        g[f"anticov_{b}_count"], g[f"anticov_{b}"] = ref[0, 0], D(canon(_rows(ref, 0, 16)))
    return g


if __name__ == "__main__":
    if sys.argv[1:2] == ["host"]:
        dst = ROOT / "tests" / "golden" / "oracle_vs_ref.npz"
        g = host()
    else:
        dst = Path(sys.argv[2]) / "ref_kernels.npz"
        g = device()
    np.savez_compressed(dst, **g)
    print(dst, dst.stat().st_size, "bytes,", len(g), "entries")
