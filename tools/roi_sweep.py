#!/usr/bin/env python
"""Time the RoIAlignRotated forward alone: channels-last pyramid resident, distinct bench tiles back to back (8 by
default = the measurement behind bench.py's `roofline`), CUDA events around the whole loop.

    python tools/roi_sweep.py [--reps 10] [--tiles 8]
"""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench as B  # noqa: E402
import workloads as W  # noqa: E402
from rs_detection_b200 import core  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--tiles", type=int, default=8, help="distinct tiles cycled (1: the 89 MB pyramid stays L2-resident)")
a = ap.parse_args()

dev = torch.device("cuda:0")
shapes = W.fpn_shapes()
cfg = core.make_roi_cfg(shapes, [1.0 / s for s in W.STRIDES], 7, 2, 1, B.EXTEND, 56.0, channels_last=True)
tiles = []
for t in range(a.tiles):
    fs, r, b, s = B.tile_inputs(t)
    tiles.append(([core.nchw_to_nhwc(torch.from_numpy(f).to(dev)) for f in fs], torch.from_numpy(r).to(dev)))
out = torch.empty((B.K_ROIS, W.CHANNELS, 7, 7), device=dev)


def run():
    for f, r in tiles:
        core.roi_align_rotated_forward(cfg, f, r, out=out)


for _ in range(3):
    run()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(a.reps):
    run()
e1.record()
torch.cuda.synchronize()
print(f"{e0.elapsed_time(e1) / (a.tiles * a.reps) * 1000:.1f} us per {B.K_ROIS}-RoI tile (prologue + gather kernels)",
      flush=True)
