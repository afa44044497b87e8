"""Per-kernel timeline of one replay of the bench.py v8n_b32 graph (N = 1): 4 rotating input sets, 4 steps per graph,
chain A = the letterbox launches, chain B (high priority) = scan -> NMS per step.

Every launch writes, per CTA, a %globaltimer stamp at entry and one at exit (common.cuh, TlStamp), so this reports for
each kernel the start of its first CTA and the end of its last one, and for every NMS the gap between the end of its
scan and the start of its first / last CTA (how long the CTAs waited for room on an SM).  Needs a probe build:
    python -c "from tensorrtx_b200 import build; build.build(probe=True)"                       # the library as shipped
    python -c "from tensorrtx_b200 import build; build.build(defines=('TRTX_NMS_NO_PDL',), suffix='_nopdl')"
run as   TRTX_LIB=tensorrtx_b200/lib/libtrtx_hot_probe.so python tools/step_timeline.py [--nms-threads 512|1024]
(the _nopdl build launches the NMS without programmatic dependent launch; with --nms-threads 1024 it is the step as it
ran before the half-SM kernel).  Prints the card's name and power limit with the numbers."""
import argparse
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from tensorrtx_b200 import _lib as L, synth  # noqa: E402
from tensorrtx_b200.pipeline import DetectionPipeline  # noqa: E402

KIND = {1: "scan", 2: "nms", 3: "letterbox"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nms-threads", type=int, default=0, help="trtx_yolo_params.tune_nms_threads (0 = default)")
    ap.add_argument("--replays", type=int, default=200)
    ap.add_argument("--show", type=int, default=2, help="replays printed in full (the rest only enter the medians)")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = L.load()
    if not hasattr(lib, "trtx_probe_set_timeline"):
        raise SystemExit(f"{L.LIB_PATH} is not a probe build (see the docstring)")
    lib.trtx_probe_set_timeline.argtypes = [C.c_void_p, C.c_int]
    lib.trtx_probe_timeline_record_words.restype = C.c_size_t
    words = lib.trtx_probe_timeline_record_words()
    gpu = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                          "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(f"library {Path(L.LIB_PATH).name}  nms_threads {args.nms_threads or 'default'}  gpu: {gpu}")

    B, R, G = 32, 4, 4
    pipes, heads = [], []
    for i in range(R):
        p = DetectionPipeline(B, 640, 640, 640, 640, 80, (8, 16, 32), 1000, 0.5, 0.45, dev)
        p.plugin.params.tune_nms_threads = args.nms_threads
        p.frames_dev.copy_(torch.from_numpy(synth.frames(B, seed=77 + i, h=640, w=640)))
        heads.append([torch.from_numpy(h).to(dev).contiguous() for h in synth.yolov8_heads(B, seed=i, nc=80, net_w=640, net_h=640,
                                                                                          strides=(8, 16, 32))])
        pipes.append(p)
    stream = torch.cuda.Stream(dev)
    chain_b = torch.cuda.Stream(dev, priority=-1)

    def group():  # bench.py make_group(0, 4) with N = 1
        cur = torch.cuda.current_stream(dev)
        chain_b.wait_stream(cur)
        with torch.cuda.stream(chain_b):
            for j in range(G):
                pipes[j].decode_nms_gather(heads[j], None)
        for j in range(G):
            pipes[j].pre.enqueue()
        cur.wait_stream(chain_b)

    nrec = 3 * G
    buf = torch.zeros(nrec * words, dtype=torch.int64, device=dev)
    with torch.cuda.stream(stream):
        group()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        lib.trtx_probe_set_timeline(buf.data_ptr(), nrec)
        with torch.cuda.graph(g):
            group()
        lib.trtx_probe_set_timeline(None, 0)
        for _ in range(20):
            g.replay()
        torch.cuda.synchronize()
        # back-to-back replays (what bench.py times), stamps on
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(100):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        step_us = e0.elapsed_time(e1) * 1e3 / (100 * G)
        rows = []
        for r in range(args.replays):
            buf.zero_()
            g.replay()
            torch.cuda.synchronize()
            rows.append(replay_summary(buf.view(nrec, words).cpu().numpy(), r < args.show, G))
    print(f"\nback-to-back replays (probe build, stamps on): {step_us:.2f} us per step")
    keys = rows[0].keys()
    print(f"\nmedians over {args.replays} replays (us from the replay's first CTA start):")
    for k in keys:
        v = np.array([row[k] for row in rows], dtype=np.float64)
        if k == "last chain":
            print(f"  {k:34s} chain B last in {int((v == 1).sum())} of {len(v)} replays")
        else:
            print(f"  {k:34s} {np.median(v):8.2f}   (p10 {np.percentile(v, 10):7.2f}, p90 {np.percentile(v, 90):7.2f})")


def replay_summary(rec, show, G):
    launches = []
    for r in rec:
        kind, n = int(r[0]), int(r[1])
        if kind == 0:
            continue
        st = r[2:2 + 2 * n:2].astype(np.int64)
        en = r[3:3 + 2 * n:2].astype(np.int64)
        launches.append((KIND[kind], st, en))
    t0 = min(st.min() for _, st, _ in launches)
    us = lambda t: (t - t0) / 1e3  # noqa: E731
    scans = [x for x in launches if x[0] == "scan"]
    nmss = [x for x in launches if x[0] == "nms"]
    lbs = [x for x in launches if x[0] == "letterbox"]
    assert len(scans) == len(nmss) == len(lbs) == G, [x[0] for x in launches]
    out = {}
    if show:
        print("\nstep  scan start/end   nms first/last CTA start (gap after scan end)   nms end   letterbox start/end")
    for j in range(G):
        s, n, lb = scans[j], nmss[j], lbs[j]
        s0, s1 = us(s[1].min()), us(s[2].max())
        n0, n0l, n1 = us(n[1].min()), us(n[1].max()), us(n[2].max())
        l0, l1 = us(lb[1].min()), us(lb[2].max())
        if show:
            print(f"{j:4d}  {s0:7.2f} {s1:7.2f}   {n0:7.2f} ({n0 - s1:+6.2f}) {n0l:7.2f} ({n0l - s1:+6.2f})        {n1:7.2f}   {l0:7.2f} {l1:7.2f}")
        out[f"step {j} scan"] = s1 - s0
        out[f"step {j} scan end -> first nms CTA"] = n0 - s1
        out[f"step {j} scan end -> last nms CTA"] = n0l - s1
        out[f"step {j} nms (first start -> end)"] = n1 - n0
        out[f"step {j} scan start -> nms end"] = n1 - s0
    end_b = max(us(n[2].max()) for n in nmss)
    end_a = max(us(lb[2].max()) for lb in lbs)
    out["chain B end"] = end_b
    out["chain A end"] = end_a
    out["replay span"] = max(end_a, end_b)
    out["last chain"] = 1 if end_b > end_a else 0
    if show:
        print(f"chain A (letterbox) ends {end_a:.2f}, chain B (scan -> nms) ends {end_b:.2f}: "
              f"chain {'B' if end_b > end_a else 'A'} finishes last")
    return out


if __name__ == "__main__":
    main()
