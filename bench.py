#!/usr/bin/env python
"""bench.py -- detection hot path benchmark (contract: the task statement / DESIGN.md section 6).

    python bench.py --gpus N --steps K --warmup W                      # this build (sm_100a kernels), default config v8n_b32
    python bench.py --impl reference --gpus N --steps K --warmup W     # the reference's CPU path on the host cores
    python bench.py --config {v8n_b32,v5s_b1,retina_b16,rcnn_b8} ...   # the other BASELINE.json configs (N = 1)

Default config = BASELINE.json configs[1], YOLOv8n b32 640x640.  A "step" is one pass of the hot path over one batch of 32
synthetic frames per GPU: batched letterbox pre-process of the frames + fused YoloLayer decode + NMS of the backbone's head
tensors (+ the gather of the compact detections over NVLink peer memory when N > 1).  The TensorRT backbone is not on this
path; its per-stride outputs are synthetic, seeded tensors resident in HBM (in the reference they are produced on the device
by context.enqueue and handed to the plugin as device pointers, yolov8/yolov8_det.cpp:98).

value = whole-job frames/s with inputs resident in HBM; e2e = the same step through DetectionPipeline.submit with the frames
in pinned HOST memory (H2D inside the timed region) and the compact detections copied back (D2H inside the timed region).
Both arms print the same `config` dict (same workload, same stages: pre-process + decode + NMS).

Timing: W warm-up steps, then ONE block of exactly K steps bracketed by CUDA events (barrier + synchronize on both sides);
ms_per_step = block time / K (max over ranks).  The 100 ms clock sampler only has samples inside the timed window when it
lasts long enough: pick K accordingly.  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes what the timed path computed in its last step (see dump_outputs), so that two builds can be
compared output for output: the inputs are synthetic and seeded, identical from run to run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

NET, NC, STRIDES, MAX_OUT = 640, 80, (8, 16, 32), 1000
CONFIGS = {
    # BASELINE.json configs[1] -- the headline
    "v8n_b32": {"workload": "YOLOv8n 640x640 b32/GPU: letterbox pre-process + YoloLayer decode + NMS, synthetic (SURVEY 8d), fp32 heads",
                "batch": 32, "conf": 0.5, "iou": 0.45, "metric": "end_to_end_fps_yolov8n_640_b32 (pre-process + fused decode + NMS); "
                                                                  "decode+NMS us/frame alongside"},
    # configs[0]: the reference's CPU-runnable case, single image
    "v5s_b1": {"workload": "YOLOv5s 640x640 b1: letterbox pre-process + anchor-based YoloLayer decode + NMS, synthetic, fp32 heads",
               "batch": 1, "conf": 0.5, "iou": 0.45, "metric": "end_to_end_fps_yolov5s_640_b1 (pre-process + decode + NMS)"},
    # configs[2]
    "retina_b16": {"workload": "RetinaFace-R50 640x640 b16: letterbox pre-process + Decode_TRT (landmarks) + NMS, synthetic, fp32 heads",
                   "batch": 16, "conf": 0.1, "iou": 0.4, "metric": "end_to_end_fps_retinaface_640_b16 (pre-process + decode + NMS)"},
    # configs[3] (the reference code is R50-C4: SURVEY 8d)
    "rcnn_b8": {"workload": "Faster R-CNN R50-C4 b8: RpnDecode + RpnNms + PredictorDecode + BatchedNms on synthetic head tensors "
                            "(800x1067 input, 6000 -> 1000 -> 100)", "batch": 8, "conf": 0.0, "iou": 0.5,
                "metric": "plugin_chain_fps_faster_rcnn_b8 (RpnDecode + RpnNms + PredictorDecode + BatchedNms)"},
}
ALGO_BYTES_PER_IMAGE = (4 + NC) * sum((NET // s) ** 2 for s in STRIDES) * 4  # 2 822 400 B, SURVEY 8d
LETTERBOX_BYTES_PER_IMAGE = NET * NET * 3 + 3 * NET * NET * 4                  # 6 144 000 B, SURVEY 8d
DUMP_SAMPLE = 1 << 20   # elements kept of a dumped output larger than this (a fixed, seeded sample)


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def config_dict(name: str, world: int) -> dict:
    """Identical in both arms (the driver compares it)."""
    c = CONFIGS[name]
    return {"workload": c["workload"], "config": name, "batch_per_gpu": c["batch"], "global_batch": c["batch"] * world,
            "net": [NET, NET], "num_classes": NC, "max_out": MAX_OUT, "conf_thresh": c["conf"], "nms_thresh": c["iou"],
            "stages": "plugin chain" if name == "rcnn_b8" else "pre-process + decode + NMS", "data": "synthetic, seeded (tensorrtx_b200/synth.py)"}


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# --------------------------------------------------------------------------------------------------
# clocks: nvidia-smi sampled DURING the timed regions (B200_PROFILING.md "clocks line")
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, windows):
        sm, smax, reasons, inside = [], [], set(), 0
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not any(a <= ts <= b for a, b in windows):
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            inside += 1
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": inside, "sampled": "inside the timed windows only (100 ms period)"}


class AllGpuSampler:
    """N > 1, rank 0: every GPU of the box twice a second (SM / memory clocks, GPU / HBM temperatures, power, throttle reasons), so
    that a rank that is slower than the others (run.per_rank_ms_per_step) can be told from a slow host.  Never raises."""
    Q = "index,clocks.sm,clocks.mem,temperature.gpu,temperature.memory,power.draw,clocks_event_reasons.active"

    def __init__(self):
        self.proc, self.lines = None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "500"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        try:
            for line in self.proc.stdout:
                self.lines.append((time.time(), line.strip()))
        except Exception:
            pass

    def stop(self):
        try:
            if self.proc is not None:
                self.proc.terminate()
                try:
                    self.proc.wait(timeout=2)
                except Exception:
                    self.proc.kill()
        except Exception:
            pass

    def summary(self, windows):
        try:
            per = {}
            for ts, line in list(self.lines):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7 or not any(a <= ts <= b for a, b in windows):
                    continue
                per.setdefault(f[0], []).append(f[1:])
            out = []
            for idx in sorted(per, key=lambda s: int(s) if s.isdigit() else 0):
                rows = per[idx]

                def col(k, fn):
                    v = []
                    for r in rows:
                        try:
                            v.append(float(r[k]))
                        except ValueError:
                            pass
                    return fn(v) if v else None
                out.append({"gpu": int(idx) if idx.isdigit() else idx, "sm_mhz": col(0, statistics.median), "mem_mhz": col(1, statistics.median),
                            "temp_c": col(2, max), "hbm_temp_c": col(3, max), "power_w": col(4, statistics.median),
                            "reasons": sorted({r[5] for r in rows}), "samples": len(rows)})
            return out or None
        except Exception:
            return None


# --------------------------------------------------------------------------------------------------
# CPU side: the reference's own CPU code where it exists (oracle/_ref, compiled from /root/reference: host nms()),
# the oracle's restatement where the reference only has a GPU kernel (decode), the reference's Python CPU pre-process
# (yolov8/yolov8_det_trt.py:207-253, cv2).  oracle/ is test infrastructure: only this leg and --impl reference use it.
# --------------------------------------------------------------------------------------------------
class CpuPath:
    def __init__(self, name: str):
        import numpy as np

        from oracle import oracle as O

        self.np, self.O, self.name, self.cfg = np, O, name, CONFIGS[name]
        self.lib = O.load()
        self.lib.oracle_yolov8_decode_nms_image.restype = C.c_int
        self.ref, self.ref_O0 = None, None
        stem = {"v8n_b32": "yolov8", "v5s_b1": "yolov5", "retina_b16": "retina"}.get(name)
        if stem:
            for attr, suffix in (("ref", ""), ("ref_O0", "_O0")):
                p = ROOT / "oracle" / "_ref" / f"libref_{stem}_host{suffix}.so"
                if p.exists():
                    try:
                        setattr(self, attr, C.CDLL(str(p)))
                    except OSError:
                        pass
        self.nms_kind = "reference" if self.ref is not None else "port"
        try:
            import cv2
            cv2.setNumThreads(1)  # one frame per Python thread; cv2 releases the GIL
            self.cv2 = cv2
        except Exception:
            self.cv2 = None

    # ---- stages, one frame each ----
    def preprocess(self, frame):
        """preprocess_image of the reference's Python driver (yolov8/yolov8_det_trt.py:207-253): cvtColor, resize, pad 128,
        /255, HWC->CHW.  Falls back to the oracle's warp-affine restatement when cv2 is missing."""
        np, cv2 = self.np, self.cv2
        if cv2 is None:
            return self.O.warpaffine(frame, NET, NET)
        h, w = frame.shape[:2]
        image = cv2.cvtColor(frame, cv2.COLOR_BGR2RGB)
        r_w, r_h = NET / w, NET / h
        if r_h > r_w:
            tw, th = NET, int(r_w * h)
            tx1 = tx2 = 0
            ty1 = int((NET - th) / 2)
            ty2 = NET - th - ty1
        else:
            tw, th = int(r_h * w), NET
            tx1 = int((NET - tw) / 2)
            tx2 = NET - tw - tx1
            ty1 = ty2 = 0
        image = cv2.resize(image, (tw, th))
        image = cv2.copyMakeBorder(image, ty1, ty2, tx1, tx2, cv2.BORDER_CONSTANT, None, (128, 128, 128))
        image = image.astype(np.float32)
        image /= 255.0
        return np.ascontiguousarray(np.transpose(image, [2, 0, 1]))

    def make_worker_state(self):
        np = self.np
        if self.name == "retina_b16":
            tp = self.O.retina_total_priors(NET, NET)
            return {"rows": np.zeros(1 + tp * 15, np.float32), "res": np.zeros(tp * 15, np.float32), "tp": tp}
        F = 38 if self.name == "v5s_b1" else 90
        return {"rows": np.zeros(1 + MAX_OUT * F, np.float32), "res": np.zeros(MAX_OUT * F, np.float32), "F": F}

    def decode(self, heads, b, st):
        """Restated CalDetection (the reference has no CPU decode) for image b -> plugin rows in st['rows']."""
        np, lib = self.np, self.lib
        ptrs = (C.c_void_p * 3)(*[h[b].ctypes.data for h in heads])
        g = (C.c_int * 3)(*[NET // s for s in STRIDES])
        if self.name == "v8n_b32":
            lib.oracle_yolov8_decode(ptrs, 1, 3, g, g, (C.c_int * 3)(*STRIDES), NC, 17, C.c_float(0.0), 0, 0, 0, MAX_OUT, 90,
                                     C.c_float(0.1), st["rows"].ctypes.data_as(C.c_void_p), None)
        elif self.name == "v5s_b1":
            from tensorrtx_b200 import synth
            anc = np.ascontiguousarray(np.asarray(synth.V5_ANCHORS, np.float32).reshape(-1))
            lib.oracle_yolov5_decode(ptrs, 1, 3, g, g, anc.ctypes.data_as(C.c_void_p), NC, NET, NET, 0, MAX_OUT, 38, C.c_float(0.1),
                                     st["rows"].ctypes.data_as(C.c_void_p), None)
        else:
            lib.oracle_retina_decode(ptrs, 1, NET, NET, C.c_double(0.02), st["rows"].ctypes.data_as(C.c_void_p), None)

    def nms(self, st, lib=None) -> int:
        """The reference's compiled host nms() when oracle/_ref has it, else the oracle's restatement."""
        lib = self.ref if lib is None else lib
        rows, res, c = st["rows"], st["res"], self.cfg
        if lib is not None:
            if self.name == "v8n_b32":
                return lib.ref_v8_nms(rows.ctypes.data_as(C.c_void_p), C.c_float(c["conf"]), C.c_float(c["iou"]), res.ctypes.data_as(C.c_void_p))
            if self.name == "v5s_b1":
                return lib.ref_v5_nms(rows.ctypes.data_as(C.c_void_p), C.c_float(c["conf"]), C.c_float(c["iou"]), res.ctypes.data_as(C.c_void_p))
            return lib.ref_retina_nms(rows.ctypes.data_as(C.c_void_p), C.c_float(c["iou"]), res.ctypes.data_as(C.c_void_p))
        variant, F, mr = (2, 15, st["tp"]) if self.name == "retina_b16" else ((1, 38, MAX_OUT) if self.name == "v5s_b1" else (0, 90, MAX_OUT))
        self.lib.oracle_nms.restype = C.c_int
        return self.lib.oracle_nms(variant, rows.ctypes.data_as(C.c_void_p), mr, F, C.c_double(c["conf"]), C.c_float(c["iou"]),
                                   res.ctypes.data_as(C.c_void_p), None)

    def cv2_nms(self, st) -> int:
        """Row B3: cv2.dnn.NMSBoxes(Batched) on the decoded boxes (the comparator the north star names)."""
        np, cv2 = self.np, self.cv2
        F = 15 if self.name == "retina_b16" else st["F"]
        n = int(st["rows"][0])
        n = min(n, (len(st["rows"]) - 1) // F)
        r = st["rows"][1:1 + n * F].reshape(n, F)
        if n == 0:
            return 0
        if self.name == "v5s_b1":
            boxes = np.stack([r[:, 0] - r[:, 2] / 2, r[:, 1] - r[:, 3] / 2, r[:, 2], r[:, 3]], 1)
        else:
            boxes = np.stack([r[:, 0], r[:, 1], r[:, 2] - r[:, 0], r[:, 3] - r[:, 1]], 1)
        if self.name == "retina_b16":
            keep = cv2.dnn.NMSBoxes(boxes.tolist(), r[:, 4].tolist(), float(self.cfg["conf"]), float(self.cfg["iou"]))
        else:
            keep = cv2.dnn.NMSBoxesBatched(boxes.tolist(), r[:, 4].tolist(), r[:, 5].astype(int).tolist(), float(self.cfg["conf"]),
                                           float(self.cfg["iou"]))
        return len(keep)

    # ---- one frame of each timed variant (selected by name so that worker PROCESSES can run it) ----
    def task(self, key: str, f: int, st) -> int:
        B = self.frames.shape[0]
        if key == "full":          # pre-process + decode + NMS
            self.preprocess(self.frames[f % B])
            self.decode(self.heads, f % B, st)
            return self.nms(st)
        if key == "dec_nms":
            self.decode(self.heads, f % B, st)
            return self.nms(st)
        if key in ("nms_O2", "nms_O0", "cv2nms"):
            st["rows"][:] = self.decoded[f % B]
            if key == "cv2nms":
                return self.cv2_nms(st)
            return self.nms(st, self.ref_O0 if key == "nms_O0" else self.ref)
        if key == "pre":
            self.preprocess(self.frames[f % B])
            return 0
        raise KeyError(key)

    def bind(self, heads, frames) -> None:
        """Inputs (and, for the NMS-only rows, the decoded plugin rows) the workers inherit through fork()."""
        self.heads, self.frames = heads, frames
        sts = [self.make_worker_state() for _ in range(frames.shape[0])]
        for b in range(frames.shape[0]):
            self.decode(heads, b, sts[b])
        self.decoded = [s_["rows"].copy() for s_ in sts]


_CP = None  # the CpuPath the forked workers use


def _pool_task(args):
    key, first, total, stride = args
    st = _CP.make_worker_state()
    kept = 0
    for f in range(first, total, stride):
        kept += _CP.task(key, f, st)
    return kept


class CpuRunner:
    """`workers` host PROCESSES (fork; no GIL between them), one frame at a time each.  Pools persist across calls."""

    def __init__(self, cp: CpuPath):
        global _CP
        _CP = cp
        self.cp, self.pools = cp, {}

    def run(self, key: str, total: int, workers: int):
        """-> (frames/s, kept rows)"""
        if workers <= 1:
            st = self.cp.make_worker_state()
            self.cp.task(key, 0, st)  # untimed first touch
            t0 = time.perf_counter()
            kept = sum(self.cp.task(key, f, st) for f in range(total))
            return total / (time.perf_counter() - t0), kept
        import multiprocessing as mp
        if workers not in self.pools:
            pool = mp.get_context("fork").Pool(workers)
            pool.map(_pool_task, [(key, i, workers, workers) for i in range(workers)])  # untimed: page in, bind symbols
            self.pools[workers] = pool
        pool = self.pools[workers]
        t0 = time.perf_counter()
        kept = sum(pool.map(_pool_task, [(key, i, total, workers) for i in range(workers)], chunksize=1))
        return total / (time.perf_counter() - t0), kept

    def close(self):
        for p_ in self.pools.values():
            p_.terminate()
        self.pools = {}


def cpu_inputs(name: str, seed: int = 0):
    from tensorrtx_b200 import synth
    B = CONFIGS[name]["batch"]
    if name == "v8n_b32":
        heads = synth.yolov8_heads(B, seed=seed, nc=NC, net_w=NET, net_h=NET, strides=STRIDES)
    elif name == "v5s_b1":
        heads = synth.yolov5_heads(B, seed=seed)
    else:
        heads = synth.retina_heads(B, seed=seed)
    return heads, synth.frames(B, seed=77 + seed, h=NET, w=NET)


def cpu_rows(run: CpuRunner, cores: int) -> dict:
    """BASELINE.md section 2: B1 NMS only (-O2 / -O0, 1 and 8 workers), B2 decode + NMS, B3 cv2.dnn.NMSBoxes; us/frame."""
    cp = run.cp
    B = cp.frames.shape[0]
    rows = {}
    n1, n8, w8 = max(B, 64), max(B, 8 * 32), min(8, cores)
    for label in ("O2", "O0"):
        if label == "O0" and cp.ref_O0 is None:
            continue
        rows[f"B1_nms_only_{label}_1thread_us"] = 1e6 / run.run(f"nms_{label}", n1, 1)[0]
        rows[f"B1_nms_only_{label}_8workers_us"] = 1e6 / run.run(f"nms_{label}", n8, w8)[0]
    rows["B1_kind"] = cp.nms_kind + (" (compiled from /root/reference into oracle/_ref)" if cp.ref is not None else " (oracle restatement)")
    rows["B2_decode_nms_1thread_us"] = 1e6 / run.run("dec_nms", max(B, 32), 1)[0]
    rows["B2_decode_nms_8workers_us"] = 1e6 / run.run("dec_nms", n8, w8)[0]
    rows["B2_decode_nms_all_cores_us"] = 1e6 / run.run("dec_nms", max(n8, 16 * cores), cores)[0]
    if cp.cv2 is not None:
        rows["B3_cv2_dnn_NMSBoxes_1thread_us"] = 1e6 / run.run("cv2nms", max(B, 32), 1)[0]
        rows["preprocess_cv2_1thread_us"] = 1e6 / run.run("pre", max(B, 32), 1)[0]
        rows["preprocess_cv2_all_cores_us"] = 1e6 / run.run("pre", max(n8, 16 * cores), cores)[0]
    rows["note"] = ("us per frame; multi-worker rows = one frame at a time per host PROCESS (fork), throughput-equivalent us; decode = "
                    "restated CalDetection (the reference decodes on the GPU only)")
    return rows


def rcnn_cpu(total_batches: int):
    """The four rcnn plugins restated on one host thread per image batch (the reference has no CPU path for them)."""
    import numpy as np

    from oracle import oracle as O
    from tensorrtx_b200 import synth
    B = CONFIGS["rcnn_b8"]["batch"]
    anchors = synth.rcnn_anchors()
    scores, deltas = synth.rpn_inputs(B, seed=0)
    cls_scores, box_deltas, _ = synth.predictor_inputs(B, seed=1)
    t0 = time.perf_counter()
    for _ in range(total_batches):
        s6, b6 = O.rpn_decode(scores, deltas, 800, 1067, 16.0, anchors, 6000)
        props = O.rpn_nms(s6, b6, 1000, 0.7)
        s, b, c = O.predictor_decode(cls_scores, box_deltas, props, 800, 1067, (10.0, 10.0, 5.0, 5.0))
        O.batched_nms(1, s, b, c, 100, 0.5)
    return total_batches * B / (time.perf_counter() - t0)


def cpu_baseline_subprocess(name: str) -> dict:
    """The CPU path in a fresh process (it forks worker processes, which must not inherit a CUDA context): the reference
    arm of this file on a bounded sample, with the rows of BASELINE.md section 2."""
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--config", name, "--steps", "3", "--warmup", "1",
                        "--rows"], capture_output=True, text=True, timeout=600)
    try:
        return json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception:
        return {"value": None, "unit": "frames/s", "cores": host_cores(), "kind": "port", "sample": "failed: " + r.stderr[-300:]}


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the same stages on the box's host cores (rank 0 only):
    pre-process (the reference's Python/cv2 letterbox) + decode (restated plugin kernel) + nms() (compiled reference code)."""
    if rank != 0:
        return
    name, cores = args.config, host_cores()
    cfg = CONFIGS[name]
    rows = None
    if name == "rcnn_b8":
        per_step = 1
        for _ in range(min(args.warmup, 2)):
            rcnn_cpu(1)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fps = rcnn_cpu(per_step)
        dt = time.perf_counter() - t0
        fps = per_step * cfg["batch"] * args.steps / dt
        kind, cores_used, sample, kept = "port", 1, f"{per_step} batch of 8 per step x {args.steps} steps, single thread (oracle restatement)", None
    else:
        cp = CpuPath(name)
        cp.bind(*cpu_inputs(name))
        run = CpuRunner(cp)
        # "all the host threads it can use": the affinity mask can be far larger than the CPU time the container really gets
        # (cgroup quota on a shared host), and oversubscribed workers only add overhead -- so the worker count is calibrated:
        # the candidate with the best throughput on a short sample wins
        affinity = cores
        best = (0.0, cores)
        for w in sorted({w for w in (4, 8, 16, 32, 64, affinity) if w <= affinity}):
            f, _ = run.run("full", 8 * w, w)
            if f > best[0] * 1.05:
                best = (f, w)
        cores = best[1]
        for w in list(run.pools):
            if w != cores and w != min(8, affinity):
                run.pools.pop(w).terminate()
        frames_per_step = max(cfg["batch"], 16 * cores)  # bounded sample: 16 frames per worker and step (~0.1-1 s per step)
        for _ in range(min(args.warmup, 3)):
            run.run("full", frames_per_step, cores)
        t0 = time.perf_counter()
        kept = 0
        for _ in range(args.steps):
            kept += run.run("full", frames_per_step, cores)[1]
        dt = time.perf_counter() - t0
        fps = frames_per_step * args.steps / dt
        kind = "port" if cp.nms_kind == "port" else "reference (nms + pre-process) + port (decode)"
        cores_used = cores
        sample = (f"{frames_per_step} frames/step x {args.steps} steps of the synthetic set, {cores} worker processes (calibrated; affinity "
                  f"mask {affinity}); pre-process = "
                  f"{'cv2 letterbox of yolov8_det_trt.py' if cp.cv2 is not None else 'oracle warp-affine'}, decode = restated CalDetection, "
                  f"nms = {cp.nms_kind}")
        if args.rows:
            rows = cpu_rows(run, cores)
        run.close()
    print(json.dumps({
        "impl": "reference", "metric": cfg["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(name, max(1, args.gpus)),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores_used, "kind": kind, "sample": sample,
                         **({"rows": rows} if rows else {})},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "us_per_frame": 1e6 / fps, "kept_rows": kept,
    }))


# --------------------------------------------------------------------------------------------------
# GPU side
# --------------------------------------------------------------------------------------------------
def scan_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per yolo_v8_scan_kernel launch, from the committed summary of an
    `ncu --set full` capture of THIS kernel source (profiles/scan_traffic.json records the source hash); None otherwise."""
    try:
        j = json.loads((ROOT / "profiles" / "scan_traffic.json").read_text())
        h = hashlib.sha256()
        for f in ("yolo_decode.cu", "yolo_layout.cuh", "common.cuh"):
            h.update((ROOT / "tensorrtx_b200" / "csrc" / f).read_bytes())
        if j.get("src_sha256") == h.hexdigest() and isinstance(j.get("dram_bytes_per_launch"), int) and isinstance(j.get("capture"), str):
            return j
    except Exception:
        pass
    return None


PER_RANK_MS = []   # N > 1: one list per timed block with every rank's own block time (the reported time is their maximum)


def timed_blocks(step, K, W, stream, dev, world, dist, flush=None, pre=None, run_many=None):
    """W warm-up steps (0 .. W-1), then one block of exactly K steps (W .. W+K-1); returns (ms of the block,
    [(t0, t1) wall window], 1)."""
    import torch

    def block(first):
        if pre is not None:
            pre()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True, blocking=True)
        t0 = time.time()
        e0.record(stream)
        if run_many is not None:
            run_many(first, K)
        else:
            for i in range(K):
                step(first + i)
        if flush is not None:
            flush(first + K - 1)
        e1.record(stream)
        e1.synchronize()             # blocking-sync event: the host thread SLEEPS until the block is done instead of spinning -- with 8
        torch.cuda.synchronize(dev)  # ranks spinning, the container's CPU quota (~10 cores on the GPU boxes) runs out and the launching
        t1 = time.time()             # threads get descheduled (N = 8 without any gather: 61 us per step against 55 at N = 1, 2)
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            every = torch.empty(world, dtype=t.dtype, device=dev)
            dist.all_gather_into_tensor(every, t)          # per-rank block times (reported, see PER_RANK_MS)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            PER_RANK_MS.append(every.tolist())
        return ms, (t0, t1)

    if run_many is not None:
        run_many(0, W)
    else:
        for i in range(W):
            step(i)
    if flush is not None:
        flush(W - 1)
    ms, w = block(W)
    return ms, [w], 1


def dump_outputs(out_dir, arrays: dict) -> None:
    """arrays: name -> the tensor a caller of the timed path receives, after its last timed step.  Written as
    out_dir/<name>.npy in float32; a tensor of more than DUMP_SAMPLE elements is reduced to the same DUMP_SAMPLE
    flat positions on every run (seed 0, ascending).  Compact detection buffers ([B, 1 + max_det * row] with the row count
    in column 0) are passed with their row width, and their floats past the count, which no caller reads, are zeroed."""
    import numpy as np

    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, (t, row) in arrays.items():
        a = t.detach().float().cpu().numpy()
        if row:
            a = a.copy()
            for b in range(a.shape[0]):
                a[b, 1 + int(a[b, 0]) * row:] = 0
        if a.size > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[idx]
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a, np.float32))


def time_kernel_loop(fn, n, stream, dev):
    import torch
    for i in range(5):
        fn(i)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True, blocking=True)
    e0.record(stream)
    for i in range(n):
        fn(i)
    e1.record(stream)
    e1.synchronize()   # sleep, do not spin (see timed_blocks)
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / n


def peak_hbm():
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def run_v8(args, rank, world, local_rank):
    import numpy as np  # noqa: F401
    import torch

    from tensorrtx_b200 import _lib as L
    from tensorrtx_b200 import synth
    from tensorrtx_b200.pipeline import DetectionPipeline, GatherRing, PeerGather

    cfg = CONFIGS["v8n_b32"]
    BATCH, CONF, IOU = cfg["batch"], cfg["conf"], cfg["iou"]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    # ---- synthetic inputs: `sets` distinct batches so consecutive steps never hit L2-resident data ----
    R = max(2, args.sets)
    head_dtype = L.F32 if args.head_dtype == "f32" else L.F16
    tdt = torch.float32 if head_dtype == L.F32 else torch.float16
    head_sets, frame_sets_host, heads_np0, frames_np0 = [], [], None, None
    for i in range(R):
        hn = synth.yolov8_heads(BATCH, seed=1000 * rank + i, nc=NC, net_w=NET, net_h=NET, strides=STRIDES)
        fn_ = synth.frames(BATCH, seed=77 + 1000 * rank + i, h=NET, w=NET)
        if i == 0:
            heads_np0, frames_np0 = hn, fn_
        head_sets.append([torch.from_numpy(h).to(dev).to(tdt).contiguous() for h in hn])
        frame_sets_host.append(torch.from_numpy(fn_).pin_memory())
    head_bytes = sum(h.numel() * h.element_size() for h in head_sets[0])
    assert head_dtype != L.F32 or head_bytes == BATCH * ALGO_BYTES_PER_IMAGE

    def new_pipe():
        return DetectionPipeline(BATCH, NET, NET, NET, NET, NC, STRIDES, MAX_OUT, CONF, IOU, dev, head_dtype=head_dtype)
    pipe = new_pipe()
    stream = torch.cuda.Stream(dev)
    pipes_dev = []
    for i in range(R):
        p = pipe if i == 0 else new_pipe()
        p.frames_dev.copy_(frame_sets_host[i])
        pipes_dev.append(p)

    with torch.cuda.stream(stream):
        # ---- N > 1: the gather.  Preferred: fused into the NMS kernel over NVLink peer memory (no collective kernel);
        #      fallback: one NCCL all-gather per step on a side stream as a parallel graph branch (round 1).
        peer, ring, gather_mode = None, GatherRing(world, BATCH, pipe.fused.out.shape[1], dev, slots=R), "none"
        if (world > 1 or args.force_gather) and not args.nccl_gather and not args.no_gather:
            try:
                gdepth = 1 if args.fused_gather else max(1, args.gather_depth)
                peer = PeerGather(world, rank, BATCH, pipe.fused.out.shape[1], dev, slots=2 * gdepth * max(1, min(args.graph_steps, R)))
                peer.fused = bool(args.fused_gather)
                gather_mode = ("fused into nms_kernel: NVLink peer stores + flags (trtx_gather), no collective kernel" if args.fused_gather else
                               f"one gather_copy_kernel (one CTA per image block: plain NVLink peer stores) + one gather_publish_kernel (counters, relaxed stores; the kernel boundary orders them) + one gather_wait_kernel per group of steps on a third graph chain, no system-scope fence anywhere; a group is published one replay after it was computed and awaited {gdepth - 1} replay(s) later (ring of {2 * gdepth} slot groups); no collective kernel"
                               + (" [EXPERIMENT: no in-graph waits]" if args.gather_no_wait else ""))
            except Exception as e:
                print(f"[bench] rank {rank}: peer gather unavailable ({type(e).__name__}: {e}); falling back to NCCL", file=sys.stderr)
                peer = None
            ok = torch.tensor([1 if peer is not None else 0], device=dev)
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # all ranks or none
            if int(ok.item()) == 0 and peer is not None:
                peer.close()
                peer = None
        use_ring = world > 1 and peer is None and not args.no_gather

        # ---- the device-resident step.  The letterbox of a batch and the decode + NMS of a batch's head tensors are independent
        #      chains (the TensorRT backbone sits between them and is not on this path), so a graph holds G consecutive steps
        #      as TWO concurrent chains: chain A = their G letterbox launches, chain B (high priority) = their G x (scan -> NMS
        #      [-> gather wait]) launches.  Exactly one letterbox, one scan and one NMS launch per step; per-launch gaps, kernel
        #      ramps / tails and the latency-bound NMS hide under the other chain's HBM traffic.
        G = 1 if (use_ring or (args.no_overlap and peer is None)) else max(1, min(args.graph_steps, R))
        chain_b = torch.cuda.Stream(dev, priority=-1)
        chain_c = torch.cuda.Stream(dev, priority=-1)  # N > 1: the gather's push + wait kernels (tiny: dispatched ahead of the streaming grids)

        def make_step(j):   # single step (serial / NCCL-ring modes)
            p, h, prev = pipes_dev[j], head_sets[j], pipes_dev[(j - 1) % R]

            def f():
                if use_ring:
                    ring.launch(prev.fused.out, (j - 1) % R)  # fork: detections of the previous step
                p.run_device(h, overlap=not args.no_overlap, peer_gather=peer)
                if use_ring:
                    ring.join()
            return f

        NG = 2 * gdepth if peer is not None else 1   # slot groups of the gather ring (trtx_hot.h: a slot is reused 2*depth replays later)
        # compact outputs, double-buffered by replay parity when the peer gather publishes them one replay later
        outs2 = [[p.fused.out, torch.zeros_like(p.fused.out)] for p in pipes_dev] if peer is not None else None

        def make_group(j0, n, half=0):   # steps j0 .. j0+n-1 (input sets mod R) as two (N > 1: three) concurrent chains
            def f():
                cur = torch.cuda.current_stream(dev)
                chain_b.wait_stream(cur)                     # fork
                evp = {}
                if peer is not None and not peer.fused:
                    # chain C: the gather, software-pipelined by one group -- this graph PUBLISHES the detections that the
                    # previous replay left in the OTHER half of the double-buffered compact outputs (outs2[j][1 - half % 2]; the
                    # first replay publishes an unused buffer, flush_dev() publishes the last group) into slot group `half` of
                    # the gathered buffers, then WAITS for every rank's publish of the group published gdepth - 1 replays ago.
                    # The NMS of this replay writes outs2[j][half % 2], which the previous replay's publish had finished reading
                    # before this graph started: nothing on the scan -> NMS chain waits for the gather, let alone for a peer
                    # (with a single output buffer the NMS had to wait for the publish kernel: +2.7 us per step, r02e_gather.log).
                    chain_c.wait_stream(cur)
                    with torch.cuda.stream(chain_c):   # ONE copy + ONE publish kernel and ONE wait kernel for the group's n slots
                        peer.push_many([outs2[j % R][1 - half % 2] for j in range(j0, j0 + n)], half * G, MAX_OUT, 0)
                        if not args.gather_no_wait:   # the group published gdepth - 1 replays ago (gdepth = 1: the one just published)
                            peer.wait(((half - (gdepth - 1)) % NG) * G, n=n)
                        evp[0] = True
                with torch.cuda.stream(chain_b):
                    for j in range(j0, j0 + n):
                        if peer is None:
                            pipes_dev[j % R].decode_nms_gather(head_sets[j % R], None)
                        elif peer.fused:   # publish from inside nms_kernel, wait on the same chain
                            pipes_dev[j % R].decode_nms_gather(head_sets[j % R], peer, None, half * G + (j - j0), fused_gather=True)
                        else:
                            pipes_dev[j % R].fused.enqueue_scan(BATCH, head_sets[j % R])
                            pipes_dev[j % R].fused.enqueue_nms(BATCH, head_sets[j % R], out=outs2[j % R][half % 2])
                for j in range(j0, j0 + n):
                    pipes_dev[j % R].pre.enqueue()
                cur.wait_stream(chain_b)                     # join
                if evp:
                    cur.wait_stream(chain_c)
            return f

        if use_ring:  # NCCL communicator and buffers must exist before anything is captured
            ring.launch(pipes_dev[0].fused.out, 0)
            ring.join()
            torch.cuda.synchronize(dev)
            gather_mode = "NCCL all-gather of [32, 1+1000*7] fp32 per step, overlapped with the next step as a graph branch"
        needs_flush = use_ring  # make_step() gathers the PREVIOUS step's detections
        if world > 1:
            dist.barrier()  # ranks enter the (eager warm-up + capture) steps together: the gather's wait kernel gives up after ~2 s
        group_replay, tail_replay = None, {}
        if args.no_graph and peer is None:
            dev_steps = [make_step(j) for j in range(R)]
        elif G > 1 or peer is not None:
            assert R % G == 0 or G == R
            mode = "thread_local" if world > 1 else "global"
            halves = NG   # the gather walks round its ring of slot groups from replay to replay
            groups = [[pipe.capture(make_group(j0, G, h), mode) for h in range(halves)] for j0 in range(0, R, G)]
            singles = [pipe.capture(make_group(j, 1), mode) for j in range(R)] if peer is None else None
            dev_steps = [g.replay for g in singles] if singles else None
            replays = [0]

            def replay_group(k):
                groups[k][replays[0] % halves].replay()
                replays[0] += 1
            group_replay = [lambda k=k: replay_group(k) for k in range(len(groups))]
        else:
            try:
                dg = [pipe.capture(make_step(j), "thread_local" if world > 1 else "global") for j in range(R)]
                dev_steps = [g.replay for g in dg]
            except Exception as e:  # NCCL refused to be captured: graphs for the kernels, eager collective on the side stream
                if not use_ring:
                    raise
                print(f"[bench] capturing the all-gather failed ({type(e).__name__}: {e}); eager gather", file=sys.stderr)
                torch.cuda.synchronize(dev)
                gather_mode += " (eager, not captured)"
                needs_flush = False
                dgc = [p.capture(lambda p=p, h=h: p.run_device(h, overlap=not args.no_overlap)) for p, h in zip(pipes_dev, head_sets)]

                def make_eager(j):
                    def f():
                        ring.reuse(j)
                        dgc[j].replay()
                        ring.launch(pipes_dev[j].fused.out, j)
                    return f
                dev_steps = [make_eager(j) for j in range(R)]

        def step_dev(i):
            if dev_steps is None:
                raise SystemExit("--steps and --warmup must be multiples of --graph-steps when N > 1 (the gather works on whole groups)")
            dev_steps[i % R]()

        def run_dev(first, n):
            """steps first .. first+n-1: whole groups of G steps as one graph replay each, the remainder step by step"""
            i = first
            if group_replay is not None:
                while i % G and i < first + n:
                    step_dev(i)
                    i += 1
                while i + G <= first + n:
                    group_replay[(i % R) // G]()
                    i += G
            while i < first + n:
                step_dev(i)
                i += 1

        def flush_dev(i_last):
            if needs_flush:
                ring.launch(pipes_dev[i_last % R].fused.out, i_last % R)
            if use_ring:
                ring.join()
            if peer is not None and not peer.fused and group_replay is not None:
                # the publishes are pipelined by one group: deliver the detections of the last G steps inside the timed region
                h = replays[0] % NG
                peer.push_many([outs2[j % R][1 - h % 2] for j in range(i_last - G + 1, i_last + 1)], h * G, MAX_OUT, 0)
                for d in range(NG if args.gather_no_wait else gdepth):   # everything still in flight
                    peer.wait(((h - d) % NG) * G, n=G)
                replays[0] += 1

        def step_e2e(i):
            # public API call with HOST frames: H2D (copy stream, double-buffered) + pre-process + decode + NMS + D2H
            if use_ring:
                ring.join()
            pipe.submit(frame_sets_host[i % R], head_sets[i % R], peer_gather=peer, gather_slot=i % (2 * G) if peer is not None else 0)
            if use_ring:
                ring.launch(pipe.fused.out, i % R)

        sampler = ClockSampler(local_rank)
        all_gpus = AllGpuSampler() if (rank == 0 and world > 1) else None
        if rank == 0:
            sampler.start()
            if all_gpus is not None:
                all_gpus.start()
            time.sleep(0.25)
        K, W = args.steps, args.warmup
        if peer is not None:   # whole groups only
            K, W = max(G, K // G * G), max(G, (W + G - 1) // G * G)
        ms_dev, win_dev, nb_dev = timed_blocks(step_dev, K, W, stream, dev, world, dist, flush_dev, run_many=run_dev)
        if args.dump_outputs:   # N = 1 without the gather: the last timed step (W + K - 1) wrote its set's pipeline
            last = pipes_dev[(W + K - 1) % R]
            dump_outputs(args.dump_outputs, {"detections": (last.fused.out, 7), "net_input": (last.net_input, 0)})
        per_rank_ms = None   # N > 1: every rank's own mean ms per step over the timed blocks (ms_per_step is built from the per-block maxima)
        try:
            if PER_RANK_MS:
                per_rank_ms = [round(sum(blk[r] for blk in PER_RANK_MS) / len(PER_RANK_MS) / K, 6) for r in range(world)]
        except Exception:
            per_rank_ms = None
        PER_RANK_MS.clear()
        gather_verified = None
        if peer is not None and not peer.fused and group_replay is not None and not args.gather_no_wait:
            # self-check outside the timed region: after one more group + flush, every rank's gathered buffer must hold every
            # rank's detections of that group (count + live rows; rows past the count are not cleared on the peers) -- the
            # reference copy travels through an NCCL all-gather of the local outputs
            if world > 1:
                dist.barrier()
            run_dev(0, G)
            flush_dev(G - 1)
            torch.cuda.synchronize(dev)
            h = (replays[0] - 1) % NG
            cols = pipe.fused.out.shape[1]
            gather_verified = True
            for k in range(G):
                local = outs2[k % R][1 - h % 2]
                ref = torch.empty((world * BATCH, cols), dtype=local.dtype, device=dev)
                if world > 1:
                    dist.all_gather_into_tensor(ref, local.contiguous())
                else:
                    ref.copy_(local)
                got = peer.result(h * G + k)
                live = torch.arange(cols, device=dev)[None, :] < (1 + ref[:, :1].long() * 7)
                if not (torch.equal(got[:, 0], ref[:, 0]) and torch.equal(got[live], ref[live]) and float(ref[:, 0].sum()) > 0):
                    gather_verified = False
            if world > 1:   # every rank's view
                okt = torch.tensor([1 if gather_verified else 0], device=dev)
                dist.all_reduce(okt, op=dist.ReduceOp.MIN)
                gather_verified = bool(int(okt.item()))
        ms_e2e, win_e2e, nb_e2e = timed_blocks(step_e2e, K, W, stream, dev, world, dist, (lambda i: ring.join()) if use_ring else None)
        gather_err = peer.error() if peer is not None else 0

        # ---- kernels in isolation, on the timed stream, rotating input sets (CUDA events around n launches) ----
        fused, n_iso = pipe.fused, max(K, 100)
        ms_decnms = time_kernel_loop(lambda i: fused.enqueue(BATCH, head_sets[i % R]), n_iso, stream, dev)
        scan_ms_b2b = time_kernel_loop(lambda i: fused.enqueue_scan(BATCH, head_sets[i % R]), n_iso, stream, dev)
        fused.enqueue_scan(BATCH, head_sets[0])
        nms_ms = time_kernel_loop(lambda i: fused.enqueue_nms(BATCH, head_sets[0]), n_iso, stream, dev)
        nms_gather_ms = None
        if peer is not None:   # scan + NMS with the peer stores + wait, ranks in lockstep
            if world > 1:
                dist.barrier()
            def _sg(i):
                pipe.decode_nms_gather(head_sets[i % R], peer, None, i % (2 * G), fused_gather=peer.fused)
            nms_gather_ms = time_kernel_loop(_sg, n_iso, stream, dev)
        lb_ms = time_kernel_loop(lambda i: pipes_dev[i % R].pre.enqueue(), n_iso, stream, dev)
        # the same scan launches inside ONE CUDA graph (how the step runs them): launch gaps are the graph's, not Python's
        g_scan = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_scan):
            for i in range(20):
                fused.enqueue_scan(BATCH, head_sets[i % R])
        scan_ms_graph = time_kernel_loop(lambda i: g_scan.replay(), 10, stream, dev) / 20
        if rank == 0:
            sampler.stop()
            if all_gpus is not None:
                all_gpus.stop()

    def leave():
        if world == 1:
            return
        sys.stdout.flush()
        t = threading.Timer(60.0, lambda: os._exit(0))  # never outlive the run because a peer is gone
        t.daemon = True
        t.start()
        torch.cuda.synchronize(dev)
        if dev_steps:
            dev_steps.clear()
        dist.barrier()
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)

    if rank != 0:
        leave()
        return

    peak, peak_src = peak_hbm()
    algo = head_bytes
    scan_ms = min(scan_ms_b2b, scan_ms_graph)
    achieved = algo / (scan_ms * 1e-3) / 1e9
    fps = world * BATCH * K / (ms_dev * 1e-3)
    fps_e2e = world * BATCH * K / (ms_e2e * 1e-3)
    traffic = scan_traffic() if (BATCH == 32 and head_dtype == L.F32) else None
    lb_bytes = BATCH * LETTERBOX_BYTES_PER_IMAGE
    out = {
        "metric": cfg["metric"], "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if head_dtype == L.F32 else "f16", "data": "synthetic",
        "config": config_dict("v8n_b32", world),
        "run": {"parallelism": f"dp{world}: batch-sharded, gather = {gather_mode}" if world > 1 else "single GPU",
                "l2": f"inputs rotate over {R} distinct sets ({R * head_bytes / 1e6:.0f} MB of head tensors + "
                      f"{R * BATCH * NET * NET * 3 / 1e6:.0f} MB of frames > 126 MB L2)",
                "cuda_graphs": not args.no_graph,
                "overlap": (f"{G} steps per graph as two concurrent chains: letterbox launches || (scan -> NMS) launches" if G > 1 else
                            ("letterbox || (scan -> NMS) as parallel graph branches" if not args.no_overlap else "serial")),
                "timed_blocks": {"device": nb_dev, "e2e": nb_e2e, "steps_per_block": K},
                "per_rank_ms_per_step": per_rank_ms,
                "gpus_during_device_blocks": all_gpus.summary(win_dev) if all_gpus is not None else None,
                "gather_timeouts": gather_err, "gather_verified": gather_verified,
                "backbone": "not on this path (TensorRT in the reference); head tensors are synthetic and HBM-resident"},
        "clocks": sampler.summary(win_dev + win_e2e),
        "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": pipe.h2d_bytes,
                "d2h_bytes_per_step": pipe.d2h_bytes, "ms_per_step": ms_e2e / K,
                "note": "DetectionPipeline.submit(): frames from pinned host memory (H2D on a copy stream, double-buffered) + "
                        "compact detections back to pinned host (D2H) every step; PCIe-bound",
                "h2d_gbps": pipe.h2d_bytes * K / (ms_e2e * 1e-3) / 1e9},
        # our kernels inside one timed block: letterbox + scan + nms per step; the peer gather adds copy + publish + wait per group of G
        # steps plus the same three for the flush of the last group (fused variant: the publish is inside nms_kernel, one wait per step)
        "gpu_launches": 3 * K + (0 if peer is None else (K if peer.fused else 3 * (K // G) + 3)),
        "decode_nms_us_per_frame": ms_decnms * 1e3 / BATCH,
        "decode_nms_ms_per_batch": ms_decnms,
        "kernels_us": {"letterbox": lb_ms * 1e3, "scan": scan_ms_b2b * 1e3, "scan_in_graph": scan_ms_graph * 1e3, "nms": nms_ms * 1e3,
                       **({"scan+nms+gather+wait (stream)": nms_gather_ms * 1e3, "scan+nms (stream)": ms_decnms * 1e3} if nms_gather_ms else {}),
                       "sum": (lb_ms + scan_ms_b2b + nms_ms) * 1e3, "step": ms_dev / K * 1e3},
        "roofline": {"bound": "hbm", "kernel": "yolo_v8_scan_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "peak_source": peak_src,
                     "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
                     "traffic_source": traffic["capture"] if traffic else "no ncu capture of this kernel source committed (profiles/scan_traffic.json)",
                     "algorithmic_bytes_per_launch": algo, "kernel_us": scan_ms * 1e3,
                     "how": "n scan launches (rotating input sets) on the timed stream between two CUDA events / n; the smaller of "
                            "stream launches and the same launches inside one CUDA graph (both in kernels_us)"},
        "roofline_letterbox": {"bound": "hbm", "kernel": "letterbox_unit_kernel", "achieved": lb_bytes / (lb_ms * 1e-3) / 1e9, "peak": peak,
                               "unit": "GB/s", "frac": lb_bytes / (lb_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": lb_bytes,
                               "kernel_us": lb_ms * 1e3},
    }
    if not args.no_cpu_baseline and world == 1:  # rank 0 at N=1 only (bounded sample of the same workload)
        out["cpu_baseline"] = cpu_baseline_subprocess("v8n_b32")
    print(json.dumps(out), flush=True)
    leave()


def run_other(args, local_rank):
    """v5s_b1 / retina_b16 / rcnn_b8 on one GPU: same JSON shape, device-resident value + host-buffer e2e + CPU rows."""
    import torch

    from tensorrtx_b200 import plugins as P
    from tensorrtx_b200 import synth
    from tensorrtx_b200.pipeline import DetectionPipeline, RcnnHeadChain, RetinaPipeline

    name = args.config
    cfg = CONFIGS[name]
    B = cfg["batch"]
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.Stream(dev)
    R = 4 if name != "v5s_b1" else 24   # input sets rotated so that consecutive steps read different HBM lines (v5s b1: 8.6 MB / set)
    K, W = args.steps, args.warmup
    peak, peak_src = peak_hbm()
    roof = None
    with torch.cuda.stream(stream):
        if name == "rcnn_b8":
            anchors = synth.rcnn_anchors()
            sets = []
            for i in range(R):
                s, d = synth.rpn_inputs(B, seed=i)
                cs, bd, _ = synth.predictor_inputs(B, seed=100 + i)
                host = [torch.from_numpy(x).pin_memory() for x in (s, d, cs, bd)]
                sets.append((host, [x.to(dev) for x in host]))
            chain = RcnnHeadChain(B, anchors, dev)
            graphs = [chain.capture(lambda t=t: chain.run_device(*t[1])) for t in sets]
            step_dev = lambda i: graphs[i % R].replay()  # noqa: E731
            stage = [torch.empty_like(x) for x in sets[0][1]]

            def step_e2e(i):
                for dst, src in zip(stage, sets[i % R][0]):
                    dst.copy_(src, non_blocking=True)
                fs, fb, fc = chain.run_device(*stage)
                chain.out_host[:, :, 0].copy_(fs, non_blocking=True)
                chain.out_host[:, :, 1:5].copy_(fb, non_blocking=True)
                chain.out_host[:, :, 5].copy_(fc, non_blocking=True)
            h2d = sum(x.numel() * 4 for x in sets[0][0])
            d2h = chain.d2h_bytes
            parts = {}
            t = sets[0][1]
            parts["rpn_decode"] = time_kernel_loop(lambda i: chain.p_dec.enqueue(B, [t[0], t[1]], [chain.s6, chain.b6], chain.ws), 50, stream, dev)
            parts["rpn_nms"] = time_kernel_loop(lambda i: chain.p_nms.enqueue(B, [chain.s6, chain.b6], [chain.props], chain.ws), 50, stream, dev)
            parts["predictor_decode"] = time_kernel_loop(lambda i: chain.p_pred.enqueue(B, [t[2], t[3], chain.props], [chain.ps, chain.pb, chain.pc], chain.ws), 50, stream, dev)
            parts["batched_nms"] = time_kernel_loop(lambda i: chain.p_bnms.enqueue(B, [chain.ps, chain.pb, chain.pc], [chain.fs, chain.fb, chain.fc], chain.ws), 50, stream, dev)
            kernels_us = {k: v * 1e3 for k, v in parts.items()}
            launches = 4
        else:
            if name == "v5s_b1":
                kern = [P.YoloKernel(NET // s, NET // s, a) for s, a in zip(STRIDES, synth.V5_ANCHORS)]
                mk = lambda: DetectionPipeline(B, NET, NET, NET, NET, NC, STRIDES, MAX_OUT, cfg["conf"], cfg["iou"], dev,  # noqa: E731
                                               plugin=P.YoloLayerPluginV5(NC, NET, NET, MAX_OUT, False, kern))
                heads_of = lambda i: synth.yolov5_heads(B, seed=i)  # noqa: E731
                algo_per_img = 3 * (5 + NC) * 8400 * 4
            else:
                mk = lambda: RetinaPipeline(B, NET, NET, 2048, dev)  # noqa: E731
                heads_of = lambda i: synth.retina_heads(B, seed=i)  # noqa: E731
                algo_per_img = 32 * 8400 * 4
            pipes, head_sets, frame_host = [], [], []
            for i in range(R):
                p = mk()
                f = torch.from_numpy(synth.frames(B, seed=77 + i)).pin_memory()
                p.frames_dev.copy_(f)
                pipes.append(p)
                frame_host.append(f)
                head_sets.append([torch.from_numpy(h).to(dev) for h in heads_of(i)])
            graphs = [p.capture(lambda p=p, h=h: p.run_device(h)) for p, h in zip(pipes, head_sets)]
            step_dev = lambda i: graphs[i % R].replay()  # noqa: E731
            p0 = pipes[0]
            if name == "v5s_b1":
                step_e2e = lambda i: p0.submit(frame_host[i % R], head_sets[i % R])  # noqa: E731
                dn = time_kernel_loop(lambda i: p0.fused.enqueue(B, head_sets[i % R]), 100, stream, dev)
                sc = time_kernel_loop(lambda i: p0.fused.enqueue_scan(B, head_sets[i % R]), 100, stream, dev)
                kernels_us = {"decode_nms": dn * 1e3, "scan": sc * 1e3}
                roof_kernel = "yolo_v5_scan_kernel"
            else:
                step_e2e = lambda i: p0.run(frame_host[i % R], head_sets[i % R])  # noqa: E731
                dn = time_kernel_loop(lambda i: p0.decode_nms(head_sets[i % R]), 100, stream, dev)
                sc = time_kernel_loop(lambda i: p0.plugin.enqueue(B, head_sets[i % R], [p0.rows], p0.ws), 100, stream, dev)
                kernels_us = {"decode_nms": dn * 1e3, "decode (scan + pack)": sc * 1e3}
                roof_kernel = "retina_scan_kernel (+ retina_pack_kernel)"
            lb = time_kernel_loop(lambda i: pipes[i % R].pre.enqueue(), 100, stream, dev)
            kernels_us["letterbox"] = lb * 1e3
            h2d, d2h = p0.h2d_bytes, p0.d2h_bytes
            ach = B * algo_per_img / (sc * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": roof_kernel, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "peak_source": peak_src, "traffic": None, "algorithmic_bytes_per_launch": B * algo_per_img, "kernel_us": sc * 1e3,
                    "note": "nominal bytes of SURVEY 8d: the kernel streams only the gate rows (objectness / cls) of every cell and "
                            "touches the other rows for passing anchors, so `achieved` can exceed the peak at small batch (launch-bound)"}
            launches = 3 if name == "v5s_b1" else 4
        sampler = ClockSampler(local_rank)
        sampler.start()
        time.sleep(0.25)
        ms_dev, win_dev, nb = timed_blocks(step_dev, K, W, stream, dev, 1, None)
        if args.dump_outputs:   # the last timed step, W + K - 1
            if name == "rcnn_b8":   # one chain for every input set
                dump_outputs(args.dump_outputs, {"scores": (chain.fs, 0), "boxes": (chain.fb, 0), "classes": (chain.fc, 0)})
            else:
                last = pipes[(W + K - 1) % R]
                dets = (last.fused.out, 7) if name == "v5s_b1" else (last.out, 17)
                dump_outputs(args.dump_outputs, {"detections": dets, "net_input": (last.net_input, 0)})
        ms_e2e, win_e2e, nb2 = timed_blocks(step_e2e, K, W, stream, dev, 1, None)
        sampler.stop()
    fps, fps_e2e = B * K / (ms_dev * 1e-3), B * K / (ms_e2e * 1e-3)
    out = {"metric": cfg["metric"], "value": fps, "unit": "frames/s", "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": config_dict(name, 1), "us_per_frame": ms_dev / K * 1e3 / B,
           "run": {"cuda_graphs": True, "input_sets": R, "timed_blocks": {"device": nb, "e2e": nb2, "steps_per_block": K}},
           "clocks": sampler.summary(win_dev + win_e2e),
           "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K,
                   "note": "frames (rcnn: the plugin input tensors) from pinned host memory + results back to pinned host every step"},
           "gpu_launches": launches * K, "kernels_us": kernels_us, "roofline": roof}
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline_subprocess(name)
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="graft", choices=["graft", "reference"])
    ap.add_argument("--config", default="v8n_b32", choices=sorted(CONFIGS))
    ap.add_argument("--sets", type=int, default=4, help="distinct input sets rotated to defeat the 126 MB L2")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--rows", action="store_true", help="--impl reference: also time the CPU rows B1 / B2 / B3 of BASELINE.md section 2")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of CUDA graphs")
    ap.add_argument("--head-dtype", default="f32", choices=["f32", "f16"])
    ap.add_argument("--no-overlap", action="store_true", help="letterbox, scan and NMS strictly one after another")
    ap.add_argument("--graph-steps", type=int, default=4, help="consecutive steps captured into one CUDA graph (two concurrent chains)")
    ap.add_argument("--nccl-gather", action="store_true", help="N > 1: NCCL all-gather instead of the gather fused into nms_kernel")
    ap.add_argument("--no-gather", action="store_true", help="experiment: N > 1 without any gather (upper bound of the scaling)")
    ap.add_argument("--gather-depth", type=int, default=1, help="N > 1: replays between the publish of a group and the wait for it, plus one (1 = wait in the same replay); ring of 2*depth slot groups")
    ap.add_argument("--force-gather", action="store_true", help="experiment: run the peer gather's publish + wait kernels at N = 1 too (this rank is its only peer)")
    ap.add_argument("--gather-no-wait", action="store_true", help="experiment: N > 1, publish only; the waits happen once at the end of a timed block (no flow control)")
    ap.add_argument("--fused-gather", action="store_true", help="N > 1: gather stores from inside nms_kernel + one-warp wait kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "graft" or args.gpus > 1 or _env_int("WORLD_SIZE", 1) > 1 or args.force_gather):
        ap.error("--dump-outputs: --impl graft on one GPU without the gather only")
    args.warmup = max(args.warmup, 3)

    rank, world, local_rank = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    if args.config == "v8n_b32":
        run_v8(args, rank, world, local_rank)
    elif rank == 0:
        run_other(args, local_rank)


if __name__ == "__main__":
    main()
