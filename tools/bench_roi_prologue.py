#!/usr/bin/env python3
"""The prologue of RoIAlignRotated calls -- locality order and per-RoI geometry records -- kernel by kernel.

    python tools/bench_roi_prologue.py [--out profiles/roi_prologue.json] [--reps 20]

Cases, on the benchmark's seeded tiles (4 levels, C = 256, 7x7 bins, sampling ratio 2, fp32):
  fwd_nchw_32000  the timed step's call: 8 tiles as one batch, 32 000 RoIs, NCHW maps (K > 16384: roi_prep_kernel)
  fwd_cl_4000     tile 0, 4000 RoIs, channels_last maps (roi_prep_kernel)
  fwd_nchw_4000   tile 0, 4000 RoIs, NCHW maps (transpose_prep_kernel: the pyramid transpose, order and geometry blocks)
  bwd_512         the atomic backward of the first 512 RoIs of tile 0, NCHW gradient maps (BASELINE configs[2])
  bwd_4000        the same for all 4000 RoIs
Each case is warmed up, then `--reps` calls run under torch.profiler (CUDA activity only); every kernel whose name is in
PROLOGUE is the prologue, and per case the median over calls of its summed durations is reported with each kernel's
median.  The whole call is timed separately with CUDA events, profiler off (median of `--rounds` runs of `--reps`
back-to-back calls).  `check` holds an exact integer sum of the forward output's bits and the float64 sum of the
backward's gradient maps, so that two builds can be compared on the same inputs.  The 8-tile pyramid (712 MB) does not
fit the 126 MB L2; the single-tile cases run from whatever L2 holds after their warm-up.  The card's name and power
limit are read in the same run.  Needs a GPU; there is nothing to fall back to.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
import workloads as W  # noqa: E402
from bench_roi_half import card, timed  # noqa: E402
from rs_detection_b200 import core  # noqa: E402

# prologue kernels; roi_order_kernel and roi_geometry_kernel are those of builds before the one-launch prologue, listed
# so that such a build can be measured with this script too
PROLOGUE = ("roi_prep_kernel", "transpose_prep_kernel", "roi_order_kernel", "roi_geometry_kernel")
TILES = 8


def prologue_us(fn, reps):
    """-> {kernel: [us per call]} of the prologue kernels of `reps` calls of fn."""
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        name = next((k for k in PROLOGUE if k in e.name), None)
        if name and e.device_type == torch.autograd.DeviceType.CUDA:
            per.setdefault(name, []).append(e.time_range.elapsed_us())
    for k, v in per.items():
        assert len(v) == reps, f"{k}: {len(v)} launches in {reps} calls"
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "roi_prologue.json"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    tiles_np = [bench.tile_inputs(s)[:2] for s in range(TILES)]
    shapes = W.fpn_shapes(1)
    scales = [1.0 / s for s in W.STRIDES]
    K, C = bench.K_ROIS, W.CHANNELS
    feats8 = [torch.cat([torch.from_numpy(t[0][l]) for t in tiles_np], 0).to(dev) for l in range(len(shapes))]
    rois8 = torch.cat([torch.cat([torch.full((K, 1), float(i)), torch.from_numpy(t[1])[:, 1:]], 1)
                       for i, t in enumerate(tiles_np)]).to(dev)
    cfg8 = core.make_roi_cfg([tuple(x.shape) for x in feats8], scales, 7, 2, 1, bench.EXTEND, 56.0)
    cfg1 = core.make_roi_cfg(shapes, scales, 7, 2, 1, bench.EXTEND, 56.0)
    feats1 = [torch.from_numpy(f).to(dev) for f in tiles_np[0][0]]
    feats1_cl = [x.contiguous(memory_format=torch.channels_last) for x in feats1]
    assert core.roi_maps_native(feats1_cl)
    rois1 = rois8[:K].contiguous()
    out8 = torch.empty((K * TILES, C, 7, 7), device=dev)
    out1 = torch.empty((K, C, 7, 7), device=dev)
    g = torch.randn((K, C, 7, 7), device=dev, generator=torch.Generator(device=dev).manual_seed(0))

    cases = {
        "fwd_nchw_32000": lambda: core.roi_align_rotated_forward(cfg8, feats8, rois8, out=out8),
        "fwd_cl_4000": lambda: core.roi_align_rotated_forward(cfg1, feats1_cl, rois1, out=out1),
        "fwd_nchw_4000": lambda: core.roi_align_rotated_forward(cfg1, feats1, rois1, out=out1),
        "bwd_512": lambda: core.roi_align_rotated_backward(cfg1, g[:512], rois1[:512], shapes),
        "bwd_4000": lambda: core.roi_align_rotated_backward(cfg1, g, rois1, shapes),
    }

    check = {}
    for name, fn in cases.items():
        r = fn()
        if name.startswith("fwd"):
            y = out8 if name == "fwd_nchw_32000" else out1
            check[name] = int(y.view(torch.int32).to(torch.int64).sum())
        else:
            check[name] = float(sum(x.double().sum() for x in r))
    torch.cuda.synchronize()

    res_cases = {}
    for name, fn in cases.items():
        for _ in range(3):
            fn()
        per = prologue_us(fn, a.reps)
        total = [sum(v[i] for v in per.values()) for i in range(a.reps)]
        calls = [timed(fn, a.reps) for _ in range(a.rounds)]
        res_cases[name] = {
            "prologue_us": float(np.median(total)),
            "prologue_kernels_us": {k: float(np.median(v)) for k, v in per.items()},
            "prologue_launches": len(per),
            "call_ms": float(np.median(calls)),
            "call_spread": float((max(calls) - min(calls)) / np.median(calls)),
        }
    res = {
        "what": "RoIAlignRotated prologue kernels (tools/bench_roi_prologue.py)",
        "card": card(), "torch": torch.__version__,
        "method": {"reps": a.reps, "rounds": a.rounds,
                   "prologue": "torch.profiler kernel durations, median over calls of the per-call sum",
                   "call": "CUDA events around reps back-to-back calls, median over rounds, profiler off"},
        "cases": res_cases, "check": check,
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    for name, r in res_cases.items():
        ks = "  ".join(f"{k} {v:.2f}" for k, v in r["prologue_kernels_us"].items())
        print(f"{name:>15}: prologue {r['prologue_us']:.2f} us ({ks})   call {r['call_ms']:.4f} ms")
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
