#!/usr/bin/env python3
"""RoIAlignRotated for a channels_last torch pyramid on the benchmark's workload: what the native layouts save.

    python tools/bench_roi_channels_last.py [--out profiles/roi_channels_last.json] [--rounds 7]

Forward: the benchmark's 8 tiles as one batched call (32 000 RoIs, 4 levels, C = 256, 7x7, sampling ratio 2), maps
held channels_last (logical (N, C, H, W)), fp32 and bf16 maps.  Variants:
  route        what a channels_last user paid before the library took torch layouts: `.contiguous()` of every level,
               then the NCHW call (whose first kernel is the library's NCHW -> NHWC copy);
  route_cl     the same plus `.contiguous(memory_format=torch.channels_last)` of the output, for a channels_last head;
  native       the levels passed as they are (RSDET_ROI_NHWC_MAPS), (K, C, 7, 7) output;
  native_cl    the same with a channels_last output (RSDET_ROI_NHWC_ROIS): the persistent kernel stores from registers;
  gather_nchw / gather_nhwc   the gather kernel alone (library events, `core.roi_gather_kernel_ms`) of the native call
               with either output layout.
Backward (BASELINE configs[2]: 512 RoIs of tile 0 over the 4 levels, atomic): the route (NCHW gradient maps, then
`.contiguous(memory_format=torch.channels_last)` of each, what autograd does for a channels_last leaf), native (the
library writes channels_last maps), and native with a channels_last grad_out.
Every variant is warmed up, then timed with CUDA events in `--rounds` rounds that alternate the variants; each number is
the median over rounds.  The 8-tile pyramid (712 MB fp32) does not fit the 126 MB L2.  Outputs of the variants are
checked bit for bit against the route in the timed configuration.  The card's name and power limit are read in the same
run.  Needs a GPU; there is nothing to fall back to.
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

import bench  # noqa: E402
import workloads as W  # noqa: E402
from bench_roi_half import card, timed  # noqa: E402
from rs_detection_b200 import core  # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16}
TILES = 8
CL = torch.channels_last


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "roi_channels_last.json"))
    ap.add_argument("--rounds", type=int, default=7)
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
    maps = {d: [x.to(dt).contiguous(memory_format=CL) for x in feats8] for d, dt in DT.items()}
    del feats8
    assert all(core.roi_maps_native(m) for m in maps.values())
    outs = {(d, cl): torch.empty((K * TILES, C, 7, 7), device=dev, memory_format=CL if cl else torch.contiguous_format)
            for d in DT for cl in (False, True)}

    def route(d, cl):
        def run():
            y = core.roi_align_rotated_forward(cfg8, [x.contiguous() for x in maps[d]], rois8)
            return y.contiguous(memory_format=CL) if cl else y
        return run

    def native(d, cl):
        return lambda: core.roi_align_rotated_forward(cfg8, maps[d], rois8, out=outs[(d, cl)])

    # backward: 512 RoIs of tile 0, channels_last gradient maps wanted
    cfg1 = core.make_roi_cfg(shapes, scales, 7, 2, 1, bench.EXTEND, 56.0)
    r512 = rois8[:512].contiguous()
    g = torch.randn((512, C, 7, 7), device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    g_cl = g.contiguous(memory_format=CL)

    def bwd_route():
        return [x.contiguous(memory_format=CL) for x in core.roi_align_rotated_backward(cfg1, g, r512, shapes)]

    def bwd_native(grad):
        return lambda: core.roi_align_rotated_backward(cfg1, grad, r512, shapes, memory_format=CL)

    jobs = {}
    for d in DT:
        for cl in (False, True):
            jobs[("route", d, cl)] = route(d, cl)
            jobs[("native", d, cl)] = native(d, cl)
    jobs[("bwd_route",)] = bwd_route
    jobs[("bwd_native",)] = bwd_native(g)
    jobs[("bwd_native_cl_grad",)] = bwd_native(g_cl)

    # the timed configuration computes what the route computes
    for d in DT:
        for cl in (False, True):
            want = route(d, cl)()
            got = native(d, cl)()
            assert got.is_contiguous(memory_format=CL if cl else torch.contiguous_format)
            assert torch.equal(got, want), (d, cl)
    want = bwd_route()
    for k in ("bwd_native", "bwd_native_cl_grad"):
        for x, w in zip(jobs[(k,)](), want):
            assert x.is_contiguous(memory_format=CL)
            assert float((x - w).abs().max()) <= 1e-4 * max(float(w.abs().max()), 1.0), k

    def gather(d, cl):
        return core.roi_gather_kernel_ms(cfg8, maps[d], rois8, outs[(d, cl)])

    for fn in jobs.values():
        fn()
    for d in DT:
        for cl in (False, True):
            gather(d, cl)
    torch.cuda.synchronize()
    samples = {k: [] for k in jobs}
    gsamples = {(d, cl): [] for d in DT for cl in (False, True)}
    for _ in range(a.rounds):
        for k, fn in jobs.items():
            samples[k].append(timed(fn, 8 if k[0] in ("route", "native") else 20))
        for k in gsamples:
            gsamples[k].append(float(np.median([gather(*k) for _ in range(5)])))
    med = {k: float(np.median(v)) for k, v in samples.items()}
    spread = {k: float((max(v) - min(v)) / np.median(v)) for k, v in samples.items()}
    gmed = {k: float(np.median(v)) for k, v in gsamples.items()}
    gspread = {k: float((max(v) - min(v)) / np.median(v)) for k, v in gsamples.items()}

    fwd = []
    for d in DT:
        row = {"maps": d, "route_ms": med[("route", d, False)], "route_cl_ms": med[("route", d, True)],
               "native_ms": med[("native", d, False)], "native_cl_ms": med[("native", d, True)],
               "gather_nchw_out_ms": gmed[(d, False)], "gather_nhwc_out_ms": gmed[(d, True)],
               "spread": {"route": spread[("route", d, False)], "route_cl": spread[("route", d, True)],
                          "native": spread[("native", d, False)], "native_cl": spread[("native", d, True)],
                          "gather_nchw_out": gspread[(d, False)], "gather_nhwc_out": gspread[(d, True)]}}
        row["native_speedup_vs_route"] = row["route_ms"] / row["native_ms"]
        row["native_cl_speedup_vs_route_cl"] = row["route_cl_ms"] / row["native_cl_ms"]
        row["gather_nhwc_vs_nchw_out"] = row["gather_nhwc_out_ms"] / row["gather_nchw_out_ms"]
        fwd.append(row)
    bwd = {"route_ms": med[("bwd_route",)], "native_ms": med[("bwd_native",)],
           "native_cl_grad_ms": med[("bwd_native_cl_grad",)],
           "spread": {k[0]: spread[k] for k in samples if k[0].startswith("bwd")}}
    res = {
        "what": "RoIAlignRotated with a channels_last torch pyramid: the contiguous route against native layouts "
                "(tools/bench_roi_channels_last.py)",
        "card": card(), "torch": torch.__version__,
        "workload": {"tiles": TILES, "rois": K * TILES, "channels": C, "levels": len(shapes), "pooled": [7, 7],
                     "sampling_ratio": 2, "backward": "512 RoIs of tile 0 over 4 levels, atomic, fp32 (BASELINE configs[2])"},
        "method": {"rounds": a.rounds, "statistic": "median over rounds; each round alternates every variant",
                   "call": "CUDA events around 8 (forward) or 20 (backward) back-to-back calls",
                   "gather": "library events around the gather kernel of one call, median of 5 per round",
                   "l2": "the 8-tile pyramid does not fit the 126 MB L2"},
        "forward": fwd, "backward": bwd,
        "native_slower_than_route": [r["maps"] for r in fwd if r["native_speedup_vs_route"] < 1.0 or
                                     r["native_cl_speedup_vs_route_cl"] < 1.0] +
                                    (["backward"] if min(bwd["native_ms"], bwd["native_cl_grad_ms"]) > bwd["route_ms"] else []),
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in fwd:
        print(f"{r['maps']:>4}: route {r['route_ms']:.4f} / cl out {r['route_cl_ms']:.4f} ms   native {r['native_ms']:.4f} / "
              f"cl out {r['native_cl_ms']:.4f} ms   gather NCHW out {r['gather_nchw_out_ms']:.4f}  NHWC out "
              f"{r['gather_nhwc_out_ms']:.4f} ms")
    print(f"bwd: route {bwd['route_ms']:.4f} ms  native {bwd['native_ms']:.4f} ms  native + cl grad_out {bwd['native_cl_grad_ms']:.4f} ms")
    print(json.dumps({"card": res["card"], "native_slower_than_route": res["native_slower_than_route"]}))


if __name__ == "__main__":
    main()
