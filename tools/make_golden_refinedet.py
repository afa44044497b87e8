"""Regenerate tests/golden/refinedet_ref.npz: what the REFERENCE's own RefineDet post-process returns on the seeded
suites of tests/test_refinedet_{cpu,gpu}.py.  Needs oracle/_ref/libref_refinedet.so (make -C oracle -f refinedet.mk
where the reference tree exists) and a CUDA device: the reference's PriorBox() and its driver glue run on the GPU.

Stored (the tests never call the reference):
  priors                     PriorBox() table, [6375, 4] float64
  <suite>_count / _digest    per image of the suite's b32 input set: row count and oracle.refinedet.rows_digest of the
                             float32 rows (x1, y1, x2, y2, score, label) the host reads (:796-813)
  <suite>_head               the first 16 rows of image 0 (float32), for diagnosis
  nms_<n>_boxes/_scores/_keep  the reference's nms() on CPU double tensors for n synthetic boxes

usage: python tools/make_golden_refinedet.py [OUT.npz]
"""
from __future__ import annotations

import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from oracle import refinedet as R  # noqa: E402
from tensorrtx_b200 import plugins  # noqa: E402

BATCH, NMS_SIZES, suite_inputs, nms_case = R.BATCH, R.NMS_SIZES, R.suite_inputs, R.nms_case


def main(out_path: Path) -> None:
    import torch

    dev = torch.device("cuda", 0)
    g = {"priors": R.ref_priors()}
    for name in R.GOLDEN_SUITES:
        t0 = time.time()
        heads, geom = suite_inputs(name)
        priors = None if geom is None else plugins.refinedet_priors(**geom).astype(np.float64)
        d = [torch.from_numpy(h).to(dev) for h in heads]
        counts, digests = [], []
        for b in range(BATCH):
            rows = R.ref_image(*[x[b] for x in d], priors=priors)
            counts.append(len(rows))
            digests.append(R.rows_digest(rows))
            if b == 0:
                g[f"{name}_head"] = R.canon_rows(rows[:16])
        g[f"{name}_count"] = np.array(counts, np.int32)
        g[f"{name}_digest"] = np.array(digests)
        print(f"{name}: rows {counts[:4]}... {time.time() - t0:.1f} s", flush=True)
    for n in NMS_SIZES:
        boxes, scores = nms_case(n)
        g[f"nms_{n}_boxes"], g[f"nms_{n}_scores"] = boxes, scores
        g[f"nms_{n}_keep"] = R.ref_nms(boxes, scores)
    out_path.parent.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(out_path, **g)
    print(f"wrote {out_path}")


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1 else ROOT / "tests" / "golden" / "refinedet_ref.npz")
