"""RefineDet post-process timing: the library's three kernels vs the reference's own post-process.

  ours       µs per batch at b1 / b8 / b32: CUDA events around graph replays of trtx_refinedet_detect_enqueue, cycling
             through SETS input sets of the default synthetic suite (6 x 28.6 MB at b32 > the 126 MB L2, so inputs come
             from HBM); each replay is one launch sequence for the whole batch.
  reference  the compiled reference post-process (oracle/_ref/libref_refinedet.so: PriorBox, decode, nms and the glue of
             refinedet.cpp:729-790), image by image, host-synchronous as in doInference; wall clock per batch.
Prints the card name and power limit read in the same run, then one JSON line per measurement.

usage: python tools/refinedet_bench.py [--ref-batches 1,8] [--replays 200]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

SETS = 6


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = [x.strip() for x in q[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,8,32")
    ap.add_argument("--ref-batches", default="1,8")
    ap.add_argument("--replays", type=int, default=300)
    args = ap.parse_args()
    import torch

    from tensorrtx_b200 import plugins as P
    from tensorrtx_b200 import synth

    dev = torch.device("cuda", 0)
    info = card()
    print(json.dumps(info), flush=True)
    post = P.RefineDetPostprocess(device=dev)
    for B in map(int, args.batches.split(",")):
        sets = [[torch.from_numpy(h).to(dev) for h in synth.refinedet_heads(B, seed=100 + i)] for i in range(SETS)]
        out = torch.empty((B, post.output_elems()), device=dev)
        ws = torch.empty(post.getWorkspaceSize(B), dtype=torch.uint8, device=dev)
        s = torch.cuda.Stream()
        graphs = []
        with torch.cuda.stream(s):
            for d in sets:
                post.enqueue(*d, out=out, workspace=ws, stream=s)
            s.synchronize()
            for d in sets:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=s):
                    post.enqueue(*d, out=out, workspace=ws, stream=s)
                graphs.append(g)
            for i in range(3 * SETS):
                graphs[i % SETS].replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for i in range(args.replays):
                graphs[i % SETS].replay()
            e1.record(s)
            e1.synchronize()
        us = e0.elapsed_time(e1) * 1000.0 / args.replays
        rows = float(out[:, 0].mean().item())
        print(json.dumps({"impl": "trtx", "batch": B, "us_per_batch": round(us, 2), "us_per_image": round(us / B, 3),
                          "replays": args.replays, "input_sets": SETS, "mean_rows": rows, **info}), flush=True)
    from oracle import refinedet as R

    R.ref_load()
    for B in map(int, args.ref_batches.split(",")):
        d = [torch.from_numpy(h).to(dev) for h in synth.refinedet_heads(B, seed=100)]
        R.ref_image(*[x[0] for x in d])  # warm-up (module loading, allocator)
        torch.cuda.synchronize()
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            for b in range(B):
                R.ref_image(*[x[b] for x in d])
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        us = float(np.median(times)) * 1e6
        print(json.dumps({"impl": "reference", "batch": B, "us_per_batch": round(us, 1), "us_per_image": round(us / B, 1),
                          "repeats": 3, **info}), flush=True)


if __name__ == "__main__":
    main()
