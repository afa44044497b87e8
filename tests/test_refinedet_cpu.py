"""RefineDet post-process (refinedet/refinedet.cpp:553-790) without a GPU: the library's host prior table, the C ABI's
argument checks, and the plain-C oracle -- all against what the reference's own code returned, stored in
tests/golden/refinedet_ref.npz by tools/make_golden_refinedet.py (PriorBox and the driver glue ran on a B200, nms() on
CPU double tensors)."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

from oracle import refinedet as R

GOLDEN = Path(__file__).resolve().parent / "golden" / "refinedet_ref.npz"


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def test_priors_equal_reference_priorbox(golden):
    from tensorrtx_b200 import plugins as P

    got = P.refinedet_priors()
    ref = golden["priors"]
    assert got.shape == ref.shape == (6375, 4)
    assert np.array_equal(got.astype(np.float64).view(np.uint64), ref.view(np.uint64))


@pytest.mark.parametrize("suite", R.GOLDEN_SUITES)
def test_oracle_equals_reference_rows(golden, suite):
    from tensorrtx_b200 import plugins as P

    heads, geom = R.suite_inputs(suite)
    priors = P.refinedet_priors(**(geom or {}))
    out, _ = R.detect(priors, *heads)
    counts = golden[f"{suite}_count"]
    assert out[:, 0].astype(np.int32).tolist() == counts.tolist()
    for b in range(R.BATCH):
        assert R.rows_digest(R.compact_rows(out, b)) == golden[f"{suite}_digest"][b], (suite, b)
    if suite == "gated_off":
        assert counts.sum() == 0
    if suite == "overflow":
        assert np.isnan(golden["overflow_head"]).any() or any(
            np.isnan(R.compact_rows(out, b)).any() for b in range(R.BATCH))


@pytest.mark.parametrize("n", R.NMS_SIZES)
def test_oracle_nms_equals_reference_nms_on_cpu_tensors(golden, n):
    boxes, scores = golden[f"nms_{n}_boxes"], golden[f"nms_{n}_scores"]
    assert np.array_equal(R.nms(boxes, scores), golden[f"nms_{n}_keep"])


def test_ties_rank_lower_prior_first():
    from tensorrtx_b200 import plugins as P

    # the top_k cut: 5 disjoint boxes with one score keep the 3 lowest indices, in index order
    boxes = np.array([[i, 0, i + 0.5, 0.5] for i in range(5)], np.float64)
    assert R.nms(boxes, np.full(5, 0.5), top_k=3).tolist() == [0, 1, 2]
    heads, _ = R.suite_inputs("ties", batch=4)
    out, idx = R.detect(P.refinedet_priors(), *heads)
    tied = 0
    for b in range(4):
        rows = R.compact_rows(out, b)
        for c in np.unique(rows[:, 5]):
            sel = rows[:, 5] == c
            s, p = rows[sel, 4], idx[b][sel]
            assert np.all(s[:-1] >= s[1:])
            eq = s[:-1] == s[1:]
            tied += int(eq.sum())
            assert np.all(p[:-1][eq] < p[1:][eq])
    assert tied > 100


def test_abi_sizeof_and_argument_errors():
    from tensorrtx_b200 import _lib as L

    lib = L.load()
    assert lib.trtx_abi_sizeof(5) == C.sizeof(L.RefineDetParams) == 40
    assert lib.trtx_abi_sizeof(99) == 0
    n = 1
    ints = (C.c_int * 1)(4)
    ar = (C.c_float * 1)(2.0)
    assert lib.trtx_refinedet_priors(32, n, ints, ints, ints, ar, None) == 48
    assert lib.trtx_refinedet_priors(32, 0, ints, ints, ints, ar, None) == 0
    assert lib.trtx_refinedet_priors(32, n, None, ints, ints, ar, None) == 0

    def params(**kw):
        p = L.RefineDetParams(num_priors=6375, num_classes=25, obj_thresh=0.01, conf_thresh=0.01, nms_thresh=0.45,
                              top_k=1000, max_out=24000)
        p.variance[0], p.variance[1] = 0.1, 0.2
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    fake = 1 << 20  # aligned, never dereferenced: every check precedes the first launch
    ws = lib.trtx_refinedet_workspace_size(C.byref(params()), 2)
    assert ws > 0
    assert lib.trtx_refinedet_workspace_size(C.byref(params(top_k=1025)), 2) == 0
    assert lib.trtx_refinedet_workspace_size(None, 2) == 0

    def run(p, batch=2, ptrs=(fake,) * 7, ws_bytes=ws):
        return lib.trtx_refinedet_detect_enqueue(C.byref(p), batch, *ptrs[:6], ptrs[6], ws_bytes, None)

    assert run(params(top_k=1025)) == L.ERR_INVALID
    assert run(params(top_k=0)) == L.ERR_INVALID
    assert run(params(num_classes=1)) == L.ERR_INVALID
    assert run(params(max_out=0)) == L.ERR_INVALID
    assert run(params(), batch=0) == L.ERR_INVALID
    assert run(params(), ptrs=(fake, fake, None, fake, fake, fake, fake)) == L.ERR_INVALID
    assert run(params(), ptrs=(fake,) * 6 + (None,)) == L.ERR_INVALID
    assert run(params(), ptrs=(fake + 4,) + (fake,) * 6) == L.ERR_INVALID  # priors not 16-byte aligned
    assert run(params(num_classes=92)) == L.ERR_UNSUPPORTED
    assert run(params(num_priors=40000)) == L.ERR_UNSUPPORTED
    assert run(params(), ws_bytes=ws - 1) == L.ERR_WORKSPACE
