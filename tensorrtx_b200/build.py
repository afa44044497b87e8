"""In-tree build of libtrtx_hot.so (sm_100a) with nvcc.

The shared library is the product: a C-ABI (include/trtx_hot.h) with no torch / Python types in
its signatures.  It is built IN-TREE (tensorrtx_b200/lib/) so that it travels to the GPU box with
the repo snapshot; it links the CUDA runtime statically, so it loads next to torch's own runtime.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIBDIR = PKG / "lib"
LIB = LIBDIR / "libtrtx_hot.so"

SOURCES = ["yolo_decode.cu", "yolo_scan_pipe.cu", "nms.cu", "retina_decode.cu", "rcnn.cu", "preprocess.cu", "mask.cu", "roi_align.cu", "calib_host.cu", "refinedet.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden",
    "--expt-relaxed-constexpr",
    "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found (needed to build libtrtx_hot.so)")


def _stamp(sources: list[Path]) -> str:
    h = hashlib.sha256()
    for f in sorted(sources + list(CSRC.glob("*.cuh")) + [ROOT / "include" / "trtx_hot.h", Path(__file__)]):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, probe: bool = False, defines: tuple = (), suffix: str = "") -> Path:
    """Compile every CUDA source for sm_100a into tensorrtx_b200/lib/libtrtx_hot.so.
    probe=True builds libtrtx_hot_probe.so instead: the same sources with -DTRTX_NMS_PROBE (clock64 phase stamps in
    nms_kernel + trtx_probe_set_nms_stamps, used by tools/nms_probe.py; per-CTA %globaltimer stamps of the scan, NMS and
    letterbox kernels + trtx_probe_set_timeline, used by tools/step_timeline.py).  `defines` + `suffix`: further experiment
    builds (tools/scan_probe.py), never loaded by the product path."""
    srcs = [CSRC / s for s in SOURCES if (CSRC / s).exists()]
    LIBDIR.mkdir(exist_ok=True)
    if defines:
        probe = True
    lib = LIBDIR / f"libtrtx_hot_probe{suffix}.so" if probe else LIB
    stamp_file = lib.with_suffix(".stamp")
    stamp = _stamp(srcs) + "|" + ",".join(defines)
    if not force and lib.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return lib
    nvcc = _nvcc()
    objs = []
    objdir = LIBDIR / (f"obj_probe{suffix}" if probe else "obj")
    objdir.mkdir(exist_ok=True)
    procs = []
    for s in srcs:
        o = objdir / (s.stem + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-I", str(ROOT / "include"), "-I", str(CSRC), "-c", str(s), "-o", str(o)]
        if probe:
            cmd.insert(1, "-DTRTX_NMS_PROBE")
            for d in defines:
                cmd.insert(1, "-D" + d)
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for s, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s.name}:\n{out}")
        if verbose and out:
            print(out)
    cmd = [nvcc, "-shared", *NVCC_FLAGS, "-o", str(lib), *map(str, objs)]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc link failed:\n{r.stdout}")
    stamp_file.write_text(stamp)
    return lib


def build_oracle() -> Path:
    """Compile the CPU oracle (test infrastructure) and, when /root/reference exists, oracle/_ref."""
    for extra in ([], ["-f", "refinedet.mk"]):
        r = subprocess.run(["make", "-C", str(ROOT / "oracle"), *extra], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                           text=True)
        if r.returncode != 0:
            raise RuntimeError(f"oracle build failed:\n{r.stdout}")
    return ROOT / "oracle" / "libtrtx_oracle.so"


if __name__ == "__main__":
    import sys

    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
