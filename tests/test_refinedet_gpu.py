"""RefineDet post-process kernels (tensorrtx_b200/csrc/refinedet.cu) on the GPU: byte-identical to the reference's own
post-process (tests/golden/refinedet_ref.npz, made on a B200 with the same CUDA fp64 exp), and against the plain-C
oracle (glibc exp: boxes to 1e-6, counts / scores / labels exact)."""
from pathlib import Path

import numpy as np
import pytest

from oracle import refinedet as R

GOLDEN = Path(__file__).resolve().parent / "golden" / "refinedet_ref.npz"
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def _run(dev, heads, geom=None, **kw):
    import torch

    from tensorrtx_b200 import plugins as P

    kw.setdefault("num_classes", heads[3].shape[2])
    post = P.RefineDetPostprocess(**(geom or {}), device=dev, **kw)
    d = [torch.from_numpy(np.ascontiguousarray(h)).to(dev) for h in heads]
    out = post.enqueue(*d)
    torch.cuda.synchronize()
    return post, d, out.cpu().numpy()


@pytest.mark.parametrize("batch", [1, 8, 32])
@pytest.mark.parametrize("suite", R.GOLDEN_SUITES)
def test_kernel_equals_reference_rows(dev, golden, suite, batch):
    heads, geom = R.suite_inputs(suite)
    _, _, out = _run(dev, [h[:batch] for h in heads], geom)
    for b in range(batch):
        assert int(out[b, 0]) == golden[f"{suite}_count"][b], (suite, b)
        assert R.rows_digest(R.compact_rows(out, b)) == golden[f"{suite}_digest"][b], (suite, b)
    if suite == "dense":  # the top_k select ran: class 1 has > 1000 candidates in every image
        ncand = ((heads[1][:batch, :, 1] > np.float32(0.01)) & (heads[3][:batch, :, 1] > np.float32(0.01))).sum(1)
        assert ncand.min() > 1000


@pytest.mark.parametrize("suite", ["default", "dense", "overflow", "geom512"])
def test_kernel_vs_oracle(dev, suite):
    heads, geom = R.suite_inputs(suite, batch=8)
    post, _, out = _run(dev, heads, geom)
    ref, _ = R.detect(post.priors_host, *heads)
    assert np.array_equal(out[:, 0], ref[:, 0])
    for b in range(8):
        g, r = R.compact_rows(out, b), R.compact_rows(ref, b)
        assert np.array_equal(g[:, 4:], r[:, 4:])  # scores and labels: the same kept sets in the same order
        assert np.allclose(g[:, :4], r[:, :4], atol=1e-6, rtol=0, equal_nan=True)


def test_ties_equal_oracle(dev):
    heads, _ = R.suite_inputs("ties", batch=8)
    post, _, out = _run(dev, heads)
    ref, _ = R.detect(post.priors_host, *heads)
    assert np.array_equal(out[:, 0], ref[:, 0])
    for b in range(8):
        g, r = R.canon_rows(R.compact_rows(out, b)), R.canon_rows(R.compact_rows(ref, b))
        assert np.array_equal(g[:, 4:], r[:, 4:])
        assert np.allclose(g[:, :4], r[:, :4], atol=1e-6, rtol=0)


def test_max_out_keeps_the_first_rows(dev):
    heads, _ = R.suite_inputs("default", batch=4)
    _, _, full = _run(dev, heads)
    _, _, cut = _run(dev, heads, max_out=100)
    assert cut.shape == (4, 1 + 100 * 7)
    for b in range(4):
        n = int(full[b, 0])
        assert n > 100
        assert int(cut[b, 0]) == 100
        assert np.array_equal(cut[b, 1:], full[b, 1:1 + 700])
    _, _, big = _run(dev, heads, max_out=30000)
    for b in range(4):
        n = int(full[b, 0])
        assert np.array_equal(big[b, :1 + n * 7], full[b, :1 + n * 7])
        assert not big[b, 1 + n * 7:].any()


def test_graph_replay_equals_eager_and_runs_are_deterministic(dev):
    import torch

    heads, _ = R.suite_inputs("dense", batch=8)
    post, d, eager = _run(dev, heads)
    again = post.enqueue(*d)
    torch.cuda.synchronize()
    assert np.array_equal(again.cpu().numpy().view(np.uint32), eager.view(np.uint32))
    out = torch.full((8, post.output_elems()), 7.0, device=dev)
    ws = torch.empty(post.getWorkspaceSize(8), dtype=torch.uint8, device=dev)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        post.enqueue(*d, out=out, workspace=ws, stream=s)  # warm-up outside capture
        g = torch.cuda.CUDAGraph()
        out.fill_(7.0)
        with torch.cuda.graph(g, stream=s):
            post.enqueue(*d, out=out, workspace=ws, stream=s)
    out.fill_(7.0)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), eager.view(np.uint32))
