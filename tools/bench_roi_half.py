#!/usr/bin/env python3
"""RoIAlignRotated with fp32, bf16 and fp16 feature pyramids on the benchmark's tiles (BASELINE configs[1]).

    python tools/bench_roi_half.py [--out profiles/roi_half.json] [--rounds 7]

Variants: feature dtype {f32, bf16, f16} x layout {NCHW, channels-last} x output {f32, the half dtype}.  For each:
  * the whole forward call (`core.roi_align_rotated_forward`) for one tile (4000 RoIs) and for the benchmark's batched
    call (8 tiles, 32 000 RoIs in one call);
  * the gather kernel alone (`core.roi_gather_kernel_ms`: events the library records around that kernel);
  * for half inputs, the route a half pyramid took before the library read it natively: cast to fp32, fp32 call
    (and, for a half output, a cast of the output).
Backward (BASELINE configs[2]): 512 RoIs of tile 0 over the 4 levels, native half against the cast route.

Algorithmic bytes of a forward launch: s_out*K*C*49 + 24*K + s_feat*C*U (U = distinct feature pixels touched, bench.py's
`touched_pixels`), against the HBM peak bench.py uses (MEASURED_PEAKS.json, else its fallback).  All variants are warmed
up, then timed in `--rounds` rounds that alternate them; each number is the median over rounds.  A single tile's
pyramid (89 MB fp32) fits the 126 MB L2, the 8-tile batch does not.  The card's name and power limit are read in the
same run.  Needs a GPU; there is nothing to fall back to.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
import workloads as W  # noqa: E402
from rs_detection_b200 import core  # noqa: E402

DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
SIZE = {"f32": 4, "bf16": 2, "f16": 2}
TILES = 8
GATHER_WAVEFRONT_SHARE = 1800 / 5300   # DESIGN.md §4.1: 3 600 of ~5 300 L1 wavefronts per RoI are gather loads; 2-byte maps halve them


def card():
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_clock_max_mhz": None}
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        pl, clk = [v.strip() for v in line.split(",")]
        info["power_limit_w"], info["sm_clock_max_mhz"] = float(pl), float(clk)
    except Exception as e:        # the numbers are still reported, without the power limit
        info["nvidia_smi_error"] = repr(e)
    return info


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "roi_half.json"))
    ap.add_argument("--rounds", type=int, default=7)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    # ---- inputs: the benchmark's seeded tiles
    tiles_np = [bench.tile_inputs(s)[:2] for s in range(TILES)]
    shapes = W.fpn_shapes(1)
    scales = [1.0 / s for s in W.STRIDES]
    K, C = bench.K_ROIS, W.CHANNELS
    feats32 = [[torch.from_numpy(f).to(dev) for f in t[0]] for t in tiles_np]
    rois = [torch.from_numpy(t[1]).to(dev) for t in tiles_np]
    feats8 = [torch.cat([feats32[i][l] for i in range(TILES)], 0) for l in range(len(shapes))]
    rois8 = torch.cat([torch.cat([torch.full((K, 1), float(i), device=dev), r[:, 1:]], 1) for i, r in enumerate(rois)])
    del feats32[1:]
    cfgs = {}
    for cl in (False, True):
        cfgs[(cl, 1)] = core.make_roi_cfg(shapes, scales, 7, 2, 1, bench.EXTEND, 56.0, channels_last=cl)
        cfgs[(cl, 8)] = core.make_roi_cfg([(TILES,) + tuple(s[1:]) for s in shapes], scales, 7, 2, 1, bench.EXTEND, 56.0,
                                          channels_last=cl)
    maps = {}
    for d, dt in DT.items():
        for cl in (False, True):
            lay = (lambda x: x.permute(0, 2, 3, 1).contiguous()) if cl else (lambda x: x.contiguous())
            maps[(d, cl, 1)] = [lay(x.to(dt)) for x in feats32[0]]
            maps[(d, cl, 8)] = [lay(x.to(dt)) for x in feats8]
    del feats8, feats32
    U1 = float(bench.touched_pixels(tiles_np[0][1]))
    U8 = float(sum(bench.touched_pixels(t[1]) for t in tiles_np))

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (bench.py)"

    def algo_bytes(d, o, n):
        return SIZE[o] * K * n * C * 49 + 24.0 * K * n + SIZE[d] * C * (U1 if n == 1 else U8)

    # ---- forward variants
    variants = []
    for d in DT:
        for cl in (False, True):
            for o in (("f32",) if d == "f32" else ("f32", d)):
                variants.append((d, cl, o))
    outs = {}
    for d, cl, o in variants:
        for n in (1, 8):
            outs[(d, cl, o, n)] = torch.empty((K * n, C, 7, 7), dtype=DT[o], device=dev)
    ro = {1: rois[0], 8: rois8}

    def fwd(d, cl, o, n):
        return lambda: core.roi_align_rotated_forward(cfgs[(cl, n)], maps[(d, cl, n)], ro[n], out=outs[(d, cl, o, n)],
                                                      out_dtype=DT[o])

    def cast_route(d, cl, o, n):          # the route before native half: cast the levels, fp32 call, cast the output
        def run():
            y = core.roi_align_rotated_forward(cfgs[(cl, n)], [x.float() for x in maps[(d, cl, n)]], ro[n])
            return y if o == "f32" else y.to(DT[o])
        return run

    def gather(d, cl, o, n):
        return core.roi_gather_kernel_ms(cfgs[(cl, n)], maps[(d, cl, n)], ro[n], outs[(d, cl, o, n)])

    # correctness spot check in the timed configuration: native == cast route, bit for bit
    for d, cl, o in variants:
        if d != "f32":
            for n in (1, 8):
                fwd(d, cl, o, n)()
                assert torch.equal(outs[(d, cl, o, n)], cast_route(d, cl, o, n)()), (d, cl, o, n)

    jobs = {}
    for d, cl, o in variants:
        for n in (1, 8):
            jobs[("call", d, cl, o, n)] = (fwd(d, cl, o, n), 20 if n == 1 else 8)
            if d != "f32":
                jobs[("cast", d, cl, o, n)] = (cast_route(d, cl, o, n), 20 if n == 1 else 8)
    # backward, configs[2]: 512 RoIs of tile 0
    r512 = rois[0][:512].contiguous()
    gen = torch.Generator(device=dev).manual_seed(0)
    g32 = torch.randn((512, C, 7, 7), device=dev, generator=gen)
    bwd_variants = [("f32", cl, "f32") for cl in (False, True)] + \
                   [(d, cl, g) for d in ("bf16", "f16") for cl in (False, True) for g in ("f32", d)]
    gouts = {g: g32.to(DT[g]) for g in DT}
    for d, cl, g in bwd_variants:
        jobs[("bwd", d, cl, g, 1)] = ((lambda d=d, cl=cl, g=g: core.roi_align_rotated_backward(
            cfgs[(cl, 1)], gouts[g], r512, shapes, feat_dtype=DT[d])), 20)
        if d != "f32":
            jobs[("bwd_cast", d, cl, g, 1)] = ((lambda d=d, cl=cl, g=g: [x.to(DT[d]) for x in core.roi_align_rotated_backward(
                cfgs[(cl, 1)], gouts[g].float(), r512, shapes)]), 20)

    for fn, reps in jobs.values():            # warm-up: every shape and workspace size
        fn()
    for d, cl, o in variants:
        for n in (1, 8):
            gather(d, cl, o, n)
    torch.cuda.synchronize()

    samples = {k: [] for k in jobs}
    gsamples = {(d, cl, o, n): [] for d, cl, o in variants for n in (1, 8)}
    for _ in range(a.rounds):
        for k, (fn, reps) in jobs.items():
            samples[k].append(timed(fn, reps))
        for k in gsamples:
            gsamples[k].append(float(np.median([gather(*k) for _ in range(5)])))
    med = {k: float(np.median(v)) for k, v in samples.items()}
    gmed = {k: float(np.median(v)) for k, v in gsamples.items()}
    spread = {k: float((max(v) - min(v)) / np.median(v)) for k, v in samples.items()}

    fwd_rows = []
    for d, cl, o in variants:
        row = {"feat": d, "layout": "nhwc" if cl else "nchw", "out": o}
        for n in (1, 8):
            tag = "1tile" if n == 1 else "8tile"
            b = algo_bytes(d, o, n)
            row[f"call_ms_{tag}"] = med[("call", d, cl, o, n)]
            row[f"call_spread_{tag}"] = spread[("call", d, cl, o, n)]
            row[f"gather_ms_{tag}"] = gmed[(d, cl, o, n)]
            row[f"algo_bytes_{tag}"] = b
            row[f"gather_hbm_frac_{tag}"] = b / (gmed[(d, cl, o, n)] * 1e-3) / 1e9 / peak
            if d != "f32":
                row[f"cast_route_ms_{tag}"] = med[("cast", d, cl, o, n)]
                row[f"speedup_vs_cast_route_{tag}"] = med[("cast", d, cl, o, n)] / med[("call", d, cl, o, n)]
            f32_gather = gmed[("f32", cl, "f32", n)]
            row[f"gather_time_fall_vs_f32_{tag}"] = 1.0 - gmed[(d, cl, o, n)] / f32_gather
        fwd_rows.append(row)
    bwd_rows = []
    for d, cl, g in bwd_variants:
        row = {"feat": d, "layout": "nhwc" if cl else "nchw", "grad_out": g, "ms": med[("bwd", d, cl, g, 1)]}
        if d != "f32":
            row["cast_route_ms"] = med[("bwd_cast", d, cl, g, 1)]
            row["speedup_vs_cast_route"] = row["cast_route_ms"] / row["ms"]
        bwd_rows.append(row)
    slower = [r for r in fwd_rows if r["feat"] != "f32" and min(r["speedup_vs_cast_route_1tile"], r["speedup_vs_cast_route_8tile"]) < 1.0]
    slower += [r for r in bwd_rows if r["feat"] != "f32" and r["speedup_vs_cast_route"] < 1.0]
    res = {
        "what": "RoIAlignRotated forward/backward with fp32, bf16 and fp16 feature pyramids (tools/bench_roi_half.py)",
        "card": card(), "torch": torch.__version__,
        "workload": {"tiles": TILES, "rois_per_tile": K, "channels": C, "levels": len(shapes), "pooled": [7, 7],
                     "sampling_ratio": 2, "touched_pixels_1tile": U1, "touched_pixels_8tile": U8,
                     "backward": "512 RoIs of tile 0 over 4 levels (BASELINE configs[2])"},
        "method": {"rounds": a.rounds, "statistic": "median over rounds; each round alternates every variant",
                   "call": "CUDA events around 20 (1 tile) or 8 (8 tiles) back-to-back calls",
                   "gather": "library events around the gather kernel of one call (roi_gather_kernel_ms), median of 5 per round",
                   "l2": "one tile's pyramid fits the 126 MB L2 and stays warm between calls; the 8-tile batch does not fit"},
        "peak_gbs": peak, "peak_source": peak_src,
        "algo_bytes_formula": "s_out*K*C*49 + 24*K + s_feat*C*U",
        "gather_wavefront_share_predicted": GATHER_WAVEFRONT_SHARE,
        "forward": fwd_rows, "backward": bwd_rows,
        "half_slower_than_cast_route": [dict((k, r[k]) for k in ("feat", "layout") if k in r) for r in slower],
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    for r in fwd_rows:
        print(f"{r['feat']:>4} {r['layout']} out={r['out']:>4}  call {r['call_ms_1tile']:.4f} / {r['call_ms_8tile']:.4f} ms  "
              f"gather {r['gather_ms_1tile']:.4f} / {r['gather_ms_8tile']:.4f} ms  frac {r['gather_hbm_frac_8tile']:.3f}  "
              + (f"cast route {r['cast_route_ms_1tile']:.4f} / {r['cast_route_ms_8tile']:.4f} ms" if r['feat'] != 'f32' else ""))
    for r in bwd_rows:
        print(f"bwd {r['feat']:>4} {r['layout']} grad={r['grad_out']:>4}  {r['ms']:.4f} ms"
              + (f"  cast route {r['cast_route_ms']:.4f} ms" if r['feat'] != 'f32' else ""))
    print(json.dumps({"card": res["card"], "slower_than_cast": res["half_slower_than_cast_route"]}))


if __name__ == "__main__":
    main()
