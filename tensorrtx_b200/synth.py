"""Seeded synthetic inputs for the hot path (SURVEY.md section 8d "Synthetic value distribution").

numpy.random.Generator(PCG64(seed)); shared by tests/, bench.py and __graft_entry__.smoke().
Background class logits ~ N(-7, 1) (sigmoid > 0.1 needs x > -2.197: ~8e-7 per logit); per image
`n_obj` planted objects (class ~U, centre ~U(image), size log-U[32,256] px): on every stride level
the cell containing the centre and its 4-neighbours get class logit ~ N(1.5, 1) and box regressions
that decode to the object box + N(0, 0.05) -> ~15 candidates per object in overlapping clusters.
"""
from __future__ import annotations

import numpy as np

V5_ANCHORS = ((10, 13, 16, 30, 33, 23), (30, 61, 62, 45, 59, 119), (116, 90, 156, 198, 373, 326))


def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.PCG64(seed))


def _plant_cells(rng, gw, gh, cx, cy, stride):
    col, row = int(cx // stride), int(cy // stride)
    cells = []
    for dc, dr in ((0, 0), (1, 0), (-1, 0), (0, 1), (0, -1)):
        c, r = col + dc, row + dr
        if 0 <= c < gw and 0 <= r < gh:
            cells.append((c, r))
    return cells


def yolov8_heads(batch: int, seed: int = 0, nc: int = 80, net_w: int = 640, net_h: int = 640,
                 strides=(8, 16, 32), n_obj: int = 64, extra: int = 0, bg_mean: float = -7.0):
    """-> list over levels of float32 [batch, 4+nc+extra, gh*gw] (yolov8 plugin input, SURVEY 8a3)."""
    rng = _rng(seed)
    C = 4 + nc + extra
    heads = []
    for s in strides:
        gw, gh = net_w // s, net_h // s
        h = rng.standard_normal((batch, C, gh * gw), dtype=np.float32)
        h[:, 4:4 + nc] += np.float32(bg_mean)
        h[:, :4] = np.abs(h[:, :4]) * 2.0 + 0.5  # ltrb distances in grid units (positive)
        heads.append(h)
    for b in range(batch):
        for _ in range(n_obj):
            cls = int(rng.integers(0, nc))
            cx, cy = rng.uniform(0, net_w), rng.uniform(0, net_h)
            size = float(np.exp(rng.uniform(np.log(32.0), np.log(256.0))))
            x1, y1, x2, y2 = cx - size / 2, cy - size / 2, cx + size / 2, cy + size / 2
            for li, s in enumerate(strides):
                gw, gh = net_w // s, net_h // s
                for (c, r) in _plant_cells(rng, gw, gh, cx, cy, s):
                    e = r * gw + c
                    ax, ay = (c + 0.5) * s, (r + 0.5) * s
                    d = np.array([(ax - x1) / s, (ay - y1) / s, (x2 - ax) / s, (y2 - ay) / s], dtype=np.float64)
                    d += rng.normal(0, 0.05, 4)
                    heads[li][b, 0:4, e] = d.astype(np.float32)
                    heads[li][b, 4 + cls, e] = np.float32(rng.normal(1.5, 1.0))
    return heads


def yolov5_heads(batch: int, seed: int = 0, nc: int = 80, net_w: int = 640, net_h: int = 640,
                 strides=(8, 16, 32), n_obj: int = 64, seg: bool = False):
    """-> list over levels of float32 [batch, 3*(5+nc(+32)), gh*gw] (yolov5 plugin input, SURVEY 8a5)."""
    rng = _rng(seed)
    ilen = 5 + nc + (32 if seg else 0)
    heads = []
    for s in strides:
        gw, gh = net_w // s, net_h // s
        h = rng.standard_normal((batch, 3, ilen, gh * gw), dtype=np.float32)
        h[:, :, 4:5 + nc] += np.float32(-7.0)  # objectness + class logits
        heads.append(h)
    for b in range(batch):
        for _ in range(n_obj):
            cls = int(rng.integers(0, nc))
            cx, cy = rng.uniform(0, net_w), rng.uniform(0, net_h)
            for li, s in enumerate(strides):
                gw, gh = net_w // s, net_h // s
                for (c, r) in _plant_cells(rng, gw, gh, cx, cy, s):
                    e = r * gw + c
                    k = int(rng.integers(0, 3))
                    heads[li][b, k, 0:4, e] = rng.normal(0, 1.0, 4).astype(np.float32)
                    heads[li][b, k, 4, e] = np.float32(rng.normal(2.0, 1.0))
                    heads[li][b, k, 5 + cls, e] = np.float32(rng.normal(1.5, 1.0))
    return [h.reshape(batch, 3 * ilen, -1) for h in heads]


def retina_heads(batch: int, seed: int = 0, in_h: int = 640, in_w: int = 640, n_obj: int = 32):
    """-> list over strides 8/16/32 of float32 [batch, 32, h*w] = [bbox 2x4 | cls 2x2 | lmk 2x10] (SURVEY 8a6)."""
    rng = _rng(seed)
    heads = []
    for s in (8, 16, 32):
        g = (in_h // s) * (in_w // s)
        h = rng.standard_normal((batch, 32, g), dtype=np.float32)
        # cls rows 8..11: (k=0: bg, face), (k=1: bg, face); background: bg logit high, face logit low
        h[:, 8] += 4.0
        h[:, 9] -= 4.0
        h[:, 10] += 4.0
        h[:, 11] -= 4.0
        heads.append(h)
    for b in range(batch):
        for _ in range(n_obj):
            cx, cy = rng.uniform(0, in_w), rng.uniform(0, in_h)
            for li, s in enumerate((8, 16, 32)):
                gw, gh = in_w // s, in_h // s
                for (c, r) in _plant_cells(rng, gw, gh, cx, cy, s):
                    e = r * gw + c
                    k = int(rng.integers(0, 2))
                    heads[li][b, 8 + 2 * k, e] = np.float32(rng.normal(-1.0, 1.0))
                    heads[li][b, 9 + 2 * k, e] = np.float32(rng.normal(2.0, 1.0))
    return heads


def yolov3_heads(batch: int, seed: int = 0, nc: int = 80, net_w: int = 608, net_h: int = 608, strides=(32, 16, 8),
                 n_obj: int = 48):
    """-> list over levels (the plugin's order: stride 32, 16, 8) of float32 [batch, 3*(5+nc), gh, gw] (yolov3-spp plugin
    input, yololayer.cu:148-160).  Planted anchors get objectness ~N(2,1) and one class ~N(1.5,1); a third of them keep a
    weak class row (so the class gate of :171 really drops rows the objectness gate alone would keep)."""
    rng = _rng(seed)
    ilen = 5 + nc
    heads = []
    for s in strides:
        gw, gh = net_w // s, net_h // s
        h = rng.standard_normal((batch, 3, ilen, gh * gw), dtype=np.float32)
        h[:, :, 4:] += np.float32(-7.0)
        h[:, :, 2:4] *= np.float32(0.5)  # w/h logits go through expf
        heads.append(h)
    for b in range(batch):
        for _ in range(n_obj):
            cls = int(rng.integers(0, nc))
            cx, cy = rng.uniform(0, net_w), rng.uniform(0, net_h)
            for li, s in enumerate(strides):
                gw, gh = net_w // s, net_h // s
                for (c, r) in _plant_cells(rng, gw, gh, cx, cy, s):
                    e = r * gw + c
                    k = int(rng.integers(0, 3))
                    heads[li][b, k, 4, e] = np.float32(rng.normal(2.0, 1.0))
                    if rng.uniform() < 2.0 / 3.0:
                        heads[li][b, k, 5 + cls, e] = np.float32(rng.normal(1.5, 1.0))
    return [h.reshape(batch, 3 * ilen, net_h // s, net_w // s) for h, s in zip(heads, strides)]


def yolo26_rows(batch: int, seed: int = 0, nc: int = 80, anchors: int = 8400, obb: bool = False, n_obj: int = 60):
    """-> float32 [batch, anchors, 4+nc(+1)]: the yolo26 head output, one row per anchor = x1,y1,x2,y2, class
    PROBABILITIES (background ~U(0, 0.05)), angle (yolo26/plugin/yololayer.cu:189-199)."""
    rng = _rng(seed)
    C = 4 + nc + (1 if obb else 0)
    x = rng.uniform(0, 0.05, (batch, anchors, C)).astype(np.float32)
    ctr = rng.uniform(0, 640, (batch, anchors, 2))
    wh = rng.uniform(8, 200, (batch, anchors, 2))
    x[..., 0:2] = (ctr - wh / 2).astype(np.float32)
    x[..., 2:4] = (ctr + wh / 2).astype(np.float32)
    if obb:
        x[..., 4 + nc] = rng.uniform(-0.78, 2.35, (batch, anchors)).astype(np.float32)
    for b in range(batch):
        for i in rng.choice(anchors, size=min(n_obj, anchors), replace=False):
            x[b, i, 4 + int(rng.integers(0, nc))] = np.float32(rng.uniform(0.2, 0.99))
    return x


def anticov_heads(batch: int, seed: int = 0, in_h: int = 640, in_w: int = 640, n_obj: int = 32):
    """-> list over strides 8/16/32 of float32 [batch, 38, h*w] = [cls 4 | bbox 2x4 | lmk 2x10 | type 6], cls / type already
    soft-maxed (retinafaceAntiCov.cpp: reshapeSoftmax), face probability of prior k at channel 2+k, mask probability at 36+k
    (retinafaceAntiCov/decode.cu:120-127,154)."""
    rng = _rng(seed)
    heads = []
    for s in (8, 16, 32):
        g = (in_h // s) * (in_w // s)
        h = rng.standard_normal((batch, 38, g)).astype(np.float32)
        h[:, 0:4] = rng.uniform(0.0, 0.3, (batch, 4, g)).astype(np.float32)
        h[:, 4:12] *= np.float32(0.5)
        h[:, 32:38] = rng.uniform(0.0, 1.0, (batch, 6, g)).astype(np.float32)
        heads.append(h)
    for b in range(batch):
        for _ in range(n_obj):
            cx, cy = rng.uniform(0, in_w), rng.uniform(0, in_h)
            for li, s in enumerate((8, 16, 32)):
                gw, gh = in_w // s, in_h // s
                for (c, r) in _plant_cells(rng, gw, gh, cx, cy, s):
                    heads[li][b, 2 + int(rng.integers(0, 2)), r * gw + c] = np.float32(rng.uniform(0.5, 1.0))
    return heads


def frames(batch: int, seed: int = 0, h: int = 640, w: int = 640):
    """-> uint8 [batch, h, w, 3] BGR frames ~U{0..255} (worst case for bilinear parity)."""
    return _rng(seed).integers(0, 256, (batch, h, w, 3), dtype=np.uint8)


def rcnn_anchors(sizes=(32, 64, 128, 256, 512), ratios=(0.5, 1.0, 2.0)):
    """GenerateAnchors, rcnn/rcnn.cpp:62-77 (float arithmetic)."""
    res = []
    for a in sizes:
        area = np.float32(a) * np.float32(a)
        for ar in ratios:
            w = np.float32(np.sqrt(np.float32(area / np.float32(ar))))
            h = np.float32(ar) * w
            res += [np.float32(-w / 2.0), np.float32(-h / 2.0), np.float32(w / 2.0), np.float32(h / 2.0)]
    return np.asarray(res, dtype=np.float32)


def rpn_inputs(batch: int, seed: int = 0, A: int = 15, H: int = 50, W: int = 67):
    """-> scores [B, A, H, W] (logits), deltas [B, A*4, H, W] (SURVEY 8a12)."""
    rng = _rng(seed)
    scores = rng.standard_normal((batch, A, H, W), dtype=np.float32) * 2.0
    deltas = rng.standard_normal((batch, A * 4, H, W), dtype=np.float32) * 0.3
    return scores, deltas


def predictor_inputs(batch: int, seed: int = 0, N: int = 1000, Ccls: int = 80, image_h: int = 800, image_w: int = 1067):
    """-> scores [B, N, C] (softmax probs), deltas [B, N*C, 4], proposals [B, N, 4] (SURVEY 8a14)."""
    rng = _rng(seed)
    logits = rng.standard_normal((batch, N, Ccls + 1), dtype=np.float32) * 3.0
    p = np.exp(logits - logits.max(-1, keepdims=True))
    p = (p / p.sum(-1, keepdims=True)).astype(np.float32)
    scores = np.ascontiguousarray(p[..., :Ccls])
    deltas = (rng.standard_normal((batch, N * Ccls, 4), dtype=np.float32) * 0.5).astype(np.float32)
    x1 = rng.uniform(0, image_w * 0.8, (batch, N)).astype(np.float32)
    y1 = rng.uniform(0, image_h * 0.8, (batch, N)).astype(np.float32)
    w = rng.uniform(16, image_w * 0.3, (batch, N)).astype(np.float32)
    h = rng.uniform(16, image_h * 0.3, (batch, N)).astype(np.float32)
    props = np.stack([x1, y1, np.minimum(x1 + w, image_w), np.minimum(y1 + h, image_h)], -1).astype(np.float32)
    return scores, deltas, props


def _softmax(x):
    e = np.exp(x - x.max(-1, keepdims=True))
    return (e / e.sum(-1, keepdims=True)).astype(np.float32)


def _untie(conf):
    """Nudge equal values of every (image, class) column of [B, P, C] up by ulps until the column has no ties."""
    for b in range(conf.shape[0]):
        for c in range(conf.shape[2]):
            col = conf[b, :, c]
            while True:
                order = np.argsort(col, kind="stable")
                s = col[order]
                dup = np.nonzero(s[1:] == s[:-1])[0] + 1
                if dup.size == 0:
                    break
                col[order[dup]] = np.nextafter(s[dup], np.float32(np.inf))
    return conf


REFINEDET_SUITES = ("default", "dense", "gated_off", "ties", "overflow")


def refinedet_heads(batch: int, seed: int = 0, num_priors: int = 6375, num_classes: int = 25, n_obj: int = 24,
                    suite: str = "default"):
    """RefineDet engine outputs (refinedet.cpp:733-736), soft-maxed like the network: -> (arm_loc [B,P,4],
    arm_conf [B,P,2], odm_loc [B,P,4], odm_conf [B,P,C]) float32.  Background-dominant: ~18 % of priors pass the
    objectness gate and ~5 % of those are candidates of a given class; per image `n_obj` planted objects (a run of 9
    consecutive priors -- 3 cells of the same map row -- with a confident class and small regressions, so that they
    overlap).  Suites: "dense" gives class 1 of every image ~2000 candidates (the top_k = 1000 select runs), "gated_off"
    puts every objectness below the gate, "ties" rounds all scores to multiples of 1/256, "overflow" sets ~2 % of the
    size regressions to +-4000 (exp overflows to inf / underflows to 0, corners become inf or NaN).  Every suite except
    "ties" is tie-free within each (image, class) column."""
    if suite not in REFINEDET_SUITES:
        raise ValueError(suite)
    rng = _rng(seed)
    B, P, C = batch, num_priors, num_classes
    arm_loc = rng.normal(0, 0.5, (B, P, 4)).astype(np.float32)
    odm_loc = rng.normal(0, 0.5, (B, P, 4)).astype(np.float32)
    arm_logit = np.stack([np.zeros((B, P)), rng.normal(-6.0, 1.5, (B, P))], -1)
    odm_logit = rng.normal(0.0, 1.0, (B, P, C))
    odm_logit[..., 0] += 6.0
    for b in range(B):
        for _ in range(n_obj):
            p0 = int(rng.integers(0, P - 9))
            c = int(rng.integers(1, C))
            sl = slice(p0, p0 + 9)
            arm_logit[b, sl, 1] = rng.normal(3.0, 1.0, 9)
            odm_logit[b, sl, c] += rng.normal(9.0, 1.0, 9)
            arm_loc[b, sl] = rng.normal(0, 0.2, (9, 4))
            odm_loc[b, sl] = rng.normal(0, 0.2, (9, 4))
    if suite == "dense":
        for b in range(B):
            sel = rng.choice(P, 2000, replace=False)
            arm_logit[b, sel, 1] = rng.normal(3.0, 1.0, sel.size)
            odm_logit[b, sel, 1] += rng.normal(7.0, 1.0, sel.size)
    arm_conf = _softmax(arm_logit)
    if suite == "gated_off":
        arm_conf[..., 1] = np.minimum(arm_conf[..., 1], np.float32(0.005))
    odm_conf = _softmax(odm_logit)
    if suite == "ties":
        odm_conf = (np.round(odm_conf * 256) / 256).astype(np.float32)
    else:
        odm_conf = _untie(odm_conf)
    if suite == "overflow":
        for loc in (arm_loc, odm_loc):
            m = rng.random((B, P, 2)) < 0.02
            loc[..., 2:][m] = np.where(rng.random(int(m.sum())) < 0.5, 4000.0, -4000.0).astype(np.float32)
    return arm_loc, arm_conf, odm_loc, odm_conf
