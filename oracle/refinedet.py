"""ctypes/numpy wrappers for RefineDet's post-process (refinedet/refinedet.cpp:553-790).

TEST AND BENCHMARK INFRASTRUCTURE ONLY, never imported by the product package:
  detect()          the plain-C fp64 restatement (liboracle_refinedet.so, built by refinedet.mk)
  ref_*()           the reference's own PriorBox / nms / driver glue, compiled by refinedet.mk into
                    _ref/libref_refinedet.so where the reference tree exists (tools/make_golden_refinedet.py,
                    tools/refinedet_bench.py); tests read their results from tests/golden/refinedet_ref.npz.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / "liboracle_refinedet.so"
REF_LIB = HERE / "_ref" / "libref_refinedet.so"
_lib = None
_ref = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB.exists() or LIB.stat().st_mtime < (HERE / "refinedet_oracle.c").stat().st_mtime:
        subprocess.run(["make", "-C", str(HERE), "-f", "refinedet.mk", str(LIB)], check=True, stdout=subprocess.DEVNULL)
    lib = C.CDLL(str(LIB))
    f = lib.oracle_refinedet_image
    f.restype = C.c_int
    f.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_float, C.c_float,
                                     C.c_void_p, C.c_void_p]
    g = lib.oracle_refinedet_nms
    g.restype = C.c_int
    g.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]
    _lib = lib
    return lib


def nms(boxes, scores, overlap=0.45, top_k=1000):
    """The restated nms() (:632-695): boxes [n,4] / scores [n] float64 -> kept indices into boxes, keep order."""
    boxes, scores = _c(boxes, np.float64), _c(scores, np.float64)
    keep = np.zeros(max(len(scores), 1), np.int64)
    n = load().oracle_refinedet_nms(boxes.ctypes.data, scores.ctypes.data, len(scores), overlap, top_k, keep.ctypes.data)
    return keep[:n].copy()


def _c(a, dt=np.float32):
    return np.ascontiguousarray(a, dtype=dt)


def detect(priors, arm_loc, arm_conf, odm_loc, odm_conf, obj_thresh=0.01, conf_thresh=0.01, nms_thresh=0.45,
           top_k=1000, max_out=None, variance=(0.1, 0.2)):
    """Batched inputs ([B,P,4], [B,P,2], [B,P,4], [B,P,C]) -> (out [B, 1 + max_out*7] f32 in the library's compact
    layout, list over images of the kept rows' prior indices)."""
    lib = load()
    priors = _c(priors)
    B, P, Cn = odm_conf.shape
    if max_out is None:
        max_out = (Cn - 1) * top_k
    out = np.zeros((B, 1 + max_out * 7), np.float32)
    idx = []
    rows = np.zeros(((Cn - 1) * top_k, 6), np.float32)
    src = np.zeros((Cn - 1) * top_k, np.int32)
    for b in range(B):
        ins = [_c(x[b]) for x in (arm_loc, arm_conf, odm_loc, odm_conf)]
        n = lib.oracle_refinedet_image(priors.ctypes.data, *[x.ctypes.data for x in ins], P, Cn, obj_thresh, conf_thresh,
                                       nms_thresh, top_k, variance[0], variance[1], rows.ctypes.data, src.ctypes.data)
        assert n >= 0
        k = min(n, max_out)
        out[b, 0] = k
        o = out[b, 1:1 + k * 7].reshape(k, 7)
        o[:, :6] = rows[:k]
        o[:, 6] = 1.0
        idx.append(src[:n].copy())
    return out, idx


# ---- the reference's own code (needs _ref/libref_refinedet.so; ref_priors / ref_image need a GPU) ----
def ref_load():
    global _ref
    if _ref is not None:
        return _ref
    import torch  # noqa: F401  -- loads the tensor library the reference build links against

    if not REF_LIB.exists():
        raise FileNotFoundError(f"{REF_LIB} is missing: build it with make -C oracle -f refinedet.mk where the reference "
                                "tree exists")
    lib = C.CDLL(str(REF_LIB))
    lib.ref_refinedet_priors.restype = C.c_int
    lib.ref_refinedet_priors.argtypes = [C.c_void_p]
    lib.ref_refinedet_nms.restype = C.c_int
    lib.ref_refinedet_nms.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]
    lib.ref_refinedet_image.restype = C.c_int
    lib.ref_refinedet_image.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.c_void_p, C.c_int]
    _ref = lib
    return lib


def ref_priors():
    """The reference's PriorBox() table, [6375, 4] float64."""
    out = np.zeros((6375, 4), np.float64)
    n = ref_load().ref_refinedet_priors(out.ctypes.data)
    assert n == 6375, n
    return out


def ref_nms(boxes, scores, overlap=0.45, top_k=1000):
    """The reference's nms() on CPU double tensors -> kept indices into boxes (keep order)."""
    boxes, scores = _c(boxes, np.float64), _c(scores, np.float64)
    keep = np.zeros(max(len(scores), 1), np.int64)
    n = ref_load().ref_refinedet_nms(boxes.ctypes.data, scores.ctypes.data, len(scores), overlap, top_k, keep.ctypes.data)
    return keep[:n].copy()


def ref_image(arm_loc, arm_conf, odm_loc, odm_conf, priors=None, cap=24000):
    """The reference's doInference post-process (:729-790) on ONE image's device tensors ([P,4], [P,2], [P,4], [P,C],
    float32 CUDA) -> rows [n, 6] float64 (x1, y1, x2, y2, score, label).  priors: [P,4] host float64, None = PriorBox()."""
    P, Cn = odm_conf.shape
    rows = np.zeros((cap, 6), np.float64)
    pp = None
    if priors is not None:
        priors = _c(priors, np.float64)
        pp = priors.ctypes.data
    n = ref_load().ref_refinedet_image(pp, P, Cn, arm_loc.data_ptr(), arm_conf.data_ptr(), odm_loc.data_ptr(),
                                       odm_conf.data_ptr(), rows.ctypes.data, cap)
    if n < 0:
        raise RuntimeError("reference post-process failed")
    assert n <= cap, n
    return rows[:n].copy()


def canon_rows(rows):
    """Detection rows as float32 with every NaN replaced by the one quiet NaN 0x7fc00000 (NaN payloads depend on the
    processor that produced them; the golden digests compare everything else bit for bit)."""
    r = np.array(rows, dtype=np.float32, copy=True)
    r[np.isnan(r)] = np.float32(np.nan)
    return r


def rows_digest(rows) -> str:
    from oracle.oracle import digest

    return digest(canon_rows(rows))


def compact_rows(out, b):
    """Rows (x1, y1, x2, y2, score, label) of image b of a compact output [B, 1 + max_out*7]."""
    n = int(out[b, 0])
    return np.asarray(out[b, 1:1 + n * 7]).reshape(n, 7)[:, :6]


# ---- the seeded suites of tests/golden/refinedet_ref.npz (tools/make_golden_refinedet.py) ----
BATCH = 32
GEOM512 = dict(image_size=512, feature_maps=(64, 32, 16, 8), steps=(8, 16, 32, 64), min_sizes=(32, 64, 128, 256),
               aspect_ratios=(2, 2, 2, 2))
# suite -> (seed, synth.refinedet_heads kwargs, prior geometry of plugins.refinedet_priors or None = the 320 model)
SUITES = {
    "default": (11, dict(suite="default"), None),
    "dense": (12, dict(suite="dense"), None),
    "gated_off": (13, dict(suite="gated_off"), None),
    "overflow": (14, dict(suite="overflow"), None),
    "geom512": (15, dict(suite="default", num_priors=16320, num_classes=21), GEOM512),
    "ties": (16, dict(suite="ties"), None),
}
GOLDEN_SUITES = ("default", "dense", "gated_off", "overflow", "geom512")  # tie-free: the reference's order is defined
NMS_SIZES = (0, 1, 5, 300, 1500)


def suite_inputs(name, batch=BATCH):
    """-> (heads, prior geometry kwargs or None)."""
    from tensorrtx_b200 import synth

    seed, kw, geom = SUITES[name]
    return synth.refinedet_heads(batch, seed=seed, **kw), geom


def nms_case(n):
    """n boxes with distinct scores for the CPU nms() comparison -> (boxes [n,4], scores [n]) float64."""
    rng = np.random.default_rng(1000 + n)
    c = rng.uniform(0, 1, (n, 2))
    wh = rng.uniform(0.02, 0.3, (n, 2))
    return np.concatenate([c - wh / 2, c + wh / 2], 1), (rng.permutation(n) + 1).astype(np.float64) / (n + 1)
