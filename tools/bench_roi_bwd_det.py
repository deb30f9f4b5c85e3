#!/usr/bin/env python3
"""The deterministic RoIAlignRotated backward against the atomic one (BASELINE configs[2], the extractor's training half).

    python tools/bench_roi_bwd_det.py [--out profiles/roi_bwd_det.json] [--rounds 7] [--trace-dir DIR]

Workloads: 512 RoIs of the benchmark's tile 0 over the 4 levels (configs[2]), and the 8 tiles x 512 RoIs in one batched
call.  Variants: layout {NCHW, channels-last} x maps {fp32, bf16} (grad_out fp32) x path {atomic, deterministic}.
  * whole-call time (`core.roi_align_rotated_backward`) from CUDA events around 20 (1 image) or 5 (8 images)
    back-to-back calls, after a warm-up of every variant; `--rounds` rounds alternate all variants, the numbers are
    medians over rounds;
  * a separate torch.profiler run (CUDA activities, 3 calls of each deterministic variant) for the per-kernel split:
    entry build, radix sort, bin-major copy of grad_out, gather, zero fill, output transpose / conversion;
  * the two paths' gradients are compared at the timed sizes, within the backward tolerance (1e-4 of the scale, plus one
    bf16 ulp for bf16 maps), and two deterministic calls must agree bit for bit.
The card's name and power limit are read in the same run.  Needs a GPU; there is nothing to fall back to.
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import workloads as W  # noqa: E402
from bench_roi_half import card, timed  # noqa: E402
from rs_detection_b200 import core  # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16}
K1 = 512
IMAGES = 8
KERNEL_GROUPS = [("entries", "roi_bwd_det_entries"), ("sort", "DeviceRadixSort"), ("grad_out_copy", "transpose_kernel<float, float, true>"),
                 ("gather", "roi_bwd_det_gather"), ("zero_fill", "memset"), ("output_pass", "transpose_kernel<float"),
                 ("output_pass", "convert_maps")]


def group_of(name):
    for g, pat in KERNEL_GROUPS:
        if pat in name or (pat == "memset" and "Memset" in name):
            return g
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "roi_bwd_det.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--trace-dir", default=None, help="where the profiler run may write (default: a temporary directory)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    tiles = [bench.tile_inputs(s)[1][:K1] for s in range(IMAGES)]
    scales = [1.0 / s for s in W.STRIDES]
    C = W.CHANNELS
    work = {}
    for n in (1, IMAGES):
        shapes = W.fpn_shapes(n)
        rois = np.concatenate([np.concatenate([np.full((K1, 1), i, np.float32), t[:, 1:]], 1) for i, t in enumerate(tiles[:n])])
        work[n] = dict(shapes=shapes, rois=torch.from_numpy(rois).to(dev),
                       g=torch.randn((K1 * n, C, 7, 7), device=dev, generator=torch.Generator(device=dev).manual_seed(n)),
                       cfg={cl: core.make_roi_cfg(shapes, scales, 7, 2, 1, bench.EXTEND, 56.0, channels_last=cl)
                            for cl in (False, True)})

    def call(n, cl, d, det):
        w = work[n]
        return lambda: core.roi_align_rotated_backward(w["cfg"][cl], w["g"], w["rois"], w["shapes"], feat_dtype=DT[d],
                                                       deterministic=det)

    variants = [(n, cl, d) for n in (1, IMAGES) for cl in (False, True) for d in DT]
    # correctness at the timed sizes
    checks = []
    for n, cl, d in variants:
        at = [x.float() for x in call(n, cl, d, False)()]
        de = [x.float() for x in call(n, cl, d, True)()]
        de2 = call(n, cl, d, True)()
        worst = 0.0
        for x, y, z in zip(at, de, de2):
            assert torch.equal(y, z.float()), f"deterministic path not reproducible: n={n} cl={cl} {d}"
            scale = float(y.abs().max()) or 1.0
            ulp = 2.0 ** -7 * y.abs() if d == "bf16" else 0.0
            err = (x - y).abs() - ulp
            worst = max(worst, float(err.max()) / scale)
        ok = worst <= 1e-4
        checks.append({"images": n, "layout": "nhwc" if cl else "nchw", "maps": d, "max_err_over_scale": worst, "ok": ok})
        assert ok, checks[-1]

    jobs = {}
    for n, cl, d in variants:
        for det in (False, True):
            jobs[(n, cl, d, det)] = (call(n, cl, d, det), 20 if n == 1 else 5)
    for fn, _ in jobs.values():
        fn()
    torch.cuda.synchronize()
    samples = {k: [] for k in jobs}
    for _ in range(a.rounds):
        for k, (fn, reps) in jobs.items():
            samples[k].append(timed(fn, reps))
    med = {k: float(np.median(v)) for k, v in samples.items()}
    spread = {k: float((max(v) - min(v)) / np.median(v)) for k, v in samples.items()}

    # per-kernel split, profiler run of its own
    trace_dir = a.trace_dir or tempfile.mkdtemp(prefix="roi_bwd_det_")
    split = {}
    from torch.profiler import ProfilerActivity, profile
    for n, cl, d in variants:
        fn = call(n, cl, d, True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
        groups = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            if t <= 0:
                continue
            g = group_of(e.key)
            groups[g] = groups.get(g, 0.0) + t / 3.0 / 1e3      # ms per call
        split[f"{n}img-{'nhwc' if cl else 'nchw'}-{d}"] = {k: round(v, 5) for k, v in sorted(groups.items())}
    rows = []
    for n, cl, d in variants:
        at, de = med[(n, cl, d, False)], med[(n, cl, d, True)]
        rows.append({"images": n, "rois": K1 * n, "layout": "nhwc" if cl else "nchw", "maps": d, "grad_out": "f32",
                     "atomic_ms": at, "deterministic_ms": de, "ratio_det_over_atomic": de / at,
                     "spread_atomic": spread[(n, cl, d, False)], "spread_deterministic": spread[(n, cl, d, True)],
                     "deterministic_kernel_ms": split[f"{n}img-{'nhwc' if cl else 'nchw'}-{d}"]})
    res = {
        "what": "RoIAlignRotated backward: deterministic (ordered sums) vs atomic path (tools/bench_roi_bwd_det.py)",
        "card": card(), "torch": torch.__version__,
        "workload": {"rois_per_image": K1, "images": [1, IMAGES], "channels": C, "levels": 4, "pooled": [7, 7],
                     "sampling_ratio": 2, "tile": W.TILE, "entries_per_roi": 49 * 4 * 4},
        "method": {"rounds": a.rounds, "statistic": "median over rounds; each round alternates every variant",
                   "call": "CUDA events around 20 (1 image) or 5 (8 images) back-to-back core.roi_align_rotated_backward calls",
                   "kernels": "torch.profiler (CUDA activities), separate run, 3 calls per variant, device time per call"},
        "checks": checks, "results": rows,
        "deterministic_never_slower": all(r["ratio_det_over_atomic"] <= 1.0 for r in rows),
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in rows:
        print(f"{r['images']} img {r['layout']} {r['maps']:>4}: atomic {r['atomic_ms']:.4f} ms  deterministic "
              f"{r['deterministic_ms']:.4f} ms  (x{r['ratio_det_over_atomic']:.2f})  {r['deterministic_kernel_ms']}")
    print(json.dumps({"card": res["card"], "never_slower": res["deterministic_never_slower"]}))


if __name__ == "__main__":
    main()
