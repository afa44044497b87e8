"""The half-SM nms_kernel (512 threads, trtx_yolo_params.tune_nms_threads = 512) against the general 1024-thread kernel
on the same scan output: compact rows and kept anchor ids must be identical bit for bit.  Also: the programmatic
launch of the NMS behind the scan survives CUDA-graph capture (a programmatic edge) and a replay equals an eager call."""
import ctypes as C

import numpy as np
import pytest
import torch

from tensorrtx_b200 import _lib as L
from tensorrtx_b200 import plugins as P
from tensorrtx_b200 import synth

pytestmark = pytest.mark.gpu


def _heads(case, B, seed):
    nc = 1 if case == "single_class_long_segment" else 80
    if case == "dense":
        h = synth.yolov8_heads(B, seed=seed)
    elif case == "background_only":
        h = synth.yolov8_heads(B, seed=seed, n_obj=0)
    elif case == "single_class_long_segment":  # one class segment of hundreds of rows: the whole-CTA chunked path
        h = synth.yolov8_heads(B, seed=seed, nc=1, n_obj=40)
    elif case == "over_1000_candidates":       # more candidates than max_out
        h = synth.yolov8_heads(B, seed=seed, n_obj=300)
    elif case == "class_conf_ties":            # logits on a 0.25 grid: many rows share (class, conf)
        h = synth.yolov8_heads(B, seed=seed, n_obj=120)
        for x in h:
            x[:, 4:] = np.round(x[:, 4:] * 4.0) / 4.0
    return nc, h


def _run(nc, heads_dev, B, dev, threads):
    plug = P.YoloLayerPlugin(nc, 17, 0.0, 640, 640, 1000, False, False, False, (8, 16, 32))
    plug.tune(nms_threads=threads)
    fused = P.FusedYoloDecodeNms(plug, B, 0.5, 0.45, device=dev)
    comp, idx = fused.enqueue(B, heads_dev)
    torch.cuda.synchronize()
    return comp.cpu().numpy(), idx.cpu().numpy()


@pytest.mark.parametrize("B", [1, 8, 32])
@pytest.mark.parametrize("case", ["dense", "background_only", "single_class_long_segment", "over_1000_candidates",
                                  "class_conf_ties"])
def test_half_sm_nms_equals_general_kernel(dev, case, B):
    nc, heads = _heads(case, B, seed=500 + B)
    hd = [torch.from_numpy(x).to(dev).contiguous() for x in heads]
    c1024, i1024 = _run(nc, hd, B, dev, 1024)
    c512, i512 = _run(nc, hd, B, dev, 512)
    c0, i0 = _run(nc, hd, B, dev, 0)
    assert c512.tobytes() == c1024.tobytes()
    assert i512.tobytes() == i1024.tobytes()
    assert c0.tobytes() == c1024.tobytes() and i0.tobytes() == i1024.tobytes()  # the default is the 1024-thread kernel
    if case == "background_only":
        assert np.all(c512[:, 0] == 0)
    else:
        assert c512[:, 0].min() > 0
    if case == "class_conf_ties":  # the inputs really tie
        for b in range(B):
            rows = c512[b, 1:1 + int(c512[b, 0]) * 7].reshape(-1, 7)
            assert len(np.unique(rows[:, [5, 4]], axis=0)) < len(rows)


def test_half_sm_nms_refuses_what_it_does_not_cover(dev):
    plug = P.YoloLayerPlugin(80, 17, 0.0, 640, 640, 1000, False, False, False, (8, 16, 32))
    plug.tune(nms_threads=512)
    hd = [torch.from_numpy(x).to(dev).contiguous() for x in synth.yolov8_heads(2, seed=3)]
    oneshot = P.FusedYoloDecodeNms(plug, 2, 0.5, 0.45, mode=L.NMS_ONESHOT, device=dev)
    with pytest.raises(Exception):
        oneshot.enqueue(2, hd)
    plug.tune(nms_threads=256)
    greedy = P.FusedYoloDecodeNms(plug, 2, 0.5, 0.45, device=dev)
    with pytest.raises(Exception):
        greedy.enqueue(2, hd)
    torch.cuda.synchronize()


def _programmatic_edges(graph) -> int:
    """Edges of type CU_GRAPH_DEPENDENCY_TYPE_PROGRAMMATIC in a captured torch graph (driver API)."""
    cu = C.CDLL("libcuda.so.1")
    raw = C.c_void_p(graph.raw_cuda_graph())

    class EdgeData(C.Structure):
        _fields_ = [("from_port", C.c_ubyte), ("to_port", C.c_ubyte), ("type", C.c_ubyte), ("reserved", C.c_ubyte * 5)]

    n = C.c_size_t(0)
    assert cu.cuGraphGetEdges_v2(raw, None, None, None, C.byref(n)) == 0
    fr, to = (C.c_void_p * max(1, n.value))(), (C.c_void_p * max(1, n.value))()
    ed = (EdgeData * max(1, n.value))()
    assert cu.cuGraphGetEdges_v2(raw, fr, to, ed, C.byref(n)) == 0
    return sum(1 for i in range(n.value) if ed[i].type == 1)


def test_pdl_launch_in_cuda_graph_equals_eager(dev):
    B = 8
    hd = [torch.from_numpy(x).to(dev).contiguous() for x in synth.yolov8_heads(B, seed=77)]
    plug = P.YoloLayerPlugin(80, 17, 0.0, 640, 640, 1000, False, False, False, (8, 16, 32))
    fused = P.FusedYoloDecodeNms(plug, B, 0.5, 0.45, device=dev)
    comp, idx = fused.enqueue(B, hd)
    torch.cuda.synchronize()
    eager = (comp.cpu().numpy().copy(), idx.cpu().numpy().copy())
    try:
        g = torch.cuda.CUDAGraph(keep_graph=True)
    except TypeError:
        g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            fused.enqueue(B, hd)
    if hasattr(g, "raw_cuda_graph"):
        try:
            n_prog = _programmatic_edges(g)
        except (OSError, RuntimeError, AttributeError):
            n_prog = None
        if n_prog is not None:
            assert n_prog == 1  # scan -> NMS
    fused.out.zero_()
    fused.idx.zero_()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert fused.out.cpu().numpy().tobytes() == eager[0].tobytes()
    assert fused.idx.cpu().numpy().tobytes() == eager[1].tobytes()
