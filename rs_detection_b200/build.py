"""Build librsdet.so in-tree with nvcc for sm_100a (no torch extension machinery, no JIT cache).

    python -m rs_detection_b200.build [--force] [--verbose]

Every translation unit is compiled with `-gencode arch=compute_100a,code=sm_100a -lineinfo`.
The IoU / NMS / transform units use `-fmad=false`: the parity target is the reference's
un-contracted float arithmetic (see csrc/rotated_iou.cuh).
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "librsdet.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default",
          "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets"]
UNITS = {
    "box_iou.cu": ["-fmad=false"],
    "nms.cu": ["-fmad=false"],
    "transforms.cu": ["-fmad=false"],
    "head.cu": ["-fmad=false"],
    "rpn.cu": ["-fmad=false"],
    "roi_align.cu": [],
    "radix_sort.cu": [],
}


def _deps():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "rsdet.h")]


def build(force: bool = False, verbose: bool = False, ptxas_info: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    newest_src = max(os.path.getmtime(p) for p in _deps())
    objs = []
    rebuilt = False
    procs = []
    for unit, extra in UNITS.items():
        src = os.path.join(CSRC, unit)
        obj = os.path.join(OBJ, unit.replace(".cu", ".o"))
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest_src:
            cmd = [NVCC, *ARCH, *COMMON, *extra, "-c", src, "-o", obj]
            if ptxas_info:
                cmd += ["-Xptxas", "-v"]
            if verbose:
                print(" ".join(cmd), flush=True)
            procs.append((unit, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
            rebuilt = True
    for unit, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {unit}")
        if (verbose or ptxas_info) and out.strip():
            print(out)
    if rebuilt or not os.path.exists(LIB):
        cmd = [NVCC, *ARCH, "-shared", "-o", LIB, *objs]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--ptxas", action="store_true", help="print register / shared-memory usage per kernel")
    a = ap.parse_args()
    print(build(a.force, a.verbose, a.ptxas))
