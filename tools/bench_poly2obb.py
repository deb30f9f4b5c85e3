#!/usr/bin/env python3
"""poly2obb (cv2.minAreaRect + le90) on the host against rsdet_poly2obb on the device, and the two-model CSV ensemble
before and after it moved to the device.

    python tools/bench_poly2obb.py [--out profiles/poly2obb.json] [--rounds 3]

Inputs: seeded jittered rotated rectangles in scene coordinates up to 15 000 px, 4 decimals, fp64 (the CSV rows'
coordinates), at 10^5, 4*10^5, 10^6 and 4*10^6 rows.  Routes, run alternately in every round:
  host          jdet.ops.bbox_transforms.poly2obb: the mirror's loop over cv2.minAreaRect (host clock)
  device        core.poly2obb on a device-resident (n, 8) tensor (CUDA events over back-to-back calls)
  device_copies numpy in, numpy out: H2D copy, core.poly2obb, D2H copy (host clock; the D2H ends in a synchronise)
The ensemble is jdet.merge.merge_csv_with_class(thr 0.625) on workloads.csv_submissions (50 images x 2 500 objects
per submission, 250 000 rows: one NMS call takes at most 2^18 rows), before (jdet.merge._grouped_nms as it was, with
the host poly2obb) and after (the device call), host clock, each call ending with its result on the host.  Every
route's output is compared bit for bit in the same run.  The card's name and power limit are read in the same run.
Needs a GPU.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import min_area_rect_oracle as MO  # noqa: E402
import workloads as W  # noqa: E402
from bench_roi_half import card, timed  # noqa: E402
from rs_detection_b200 import core  # noqa: E402
from rs_detection_b200.jdet import merge as PM  # noqa: E402
from rs_detection_b200.jdet.ops.bbox_transforms import poly2obb as host_poly2obb  # noqa: E402

SIZES = [100_000, 400_000, 1_000_000, 4_000_000]


def grouped_nms_before(dets, group, thr_per_group):
    """jdet.merge._grouped_nms before the device poly2obb: the host loop, then the same NMS call."""
    hbb = PM.obb2hbb(PM.poly2obb(dets[:, 1:9]))
    b = torch.from_numpy(np.ascontiguousarray(hbb, dtype=np.float64)).cuda()
    s = torch.from_numpy(np.ascontiguousarray(dets[:, 9], dtype=np.float64)).cuda()
    res = core.nms(PM.NMS_HBB, b, s, float(thr_per_group[0]), labels=torch.from_numpy(group.astype(np.int32)).cuda(),
                   thr_per_label=torch.tensor(thr_per_group, dtype=torch.float64, device=b.device), want_mask=False,
                   want_sorted=False, want_score=True, ws_tag="merge")
    kept = res.score_idx.cpu().numpy()
    return kept[np.argsort(group[kept], kind="stable")]


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def same(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.int64), np.ascontiguousarray(b).view(np.int64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "poly2obb.json"))
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    real_poly2obb, grouped_nms_after = core.poly2obb, PM._grouped_nms
    rows, checks = [], {}
    for n in SIZES:
        q = MO.rotated_rects(np.random.default_rng(n), n)
        qd = torch.from_numpy(q).cuda()
        ref = host_poly2obb(q)
        dev_out = real_poly2obb(qd).cpu().numpy()
        checks[f"n={n}"] = bool(same(dev_out, ref))
        reps = max(1, 20_000_000 // n)
        for _ in range(3):
            real_poly2obb(qd)
        samples = {"host": [], "device": [], "device_copies": []}
        for _ in range(a.rounds):
            samples["host"].append(wall(lambda: host_poly2obb(q))[0])
            samples["device"].append(timed(lambda: real_poly2obb(qd), reps))
            ms, out = wall(lambda: real_poly2obb(torch.from_numpy(q).cuda()).cpu().numpy())
            samples["device_copies"].append(ms)
            checks[f"n={n}"] &= bool(same(out, ref))
        row = {"rows": n, "ms": {k: float(np.median(v)) for k, v in samples.items()},
               "spread": {k: float((max(v) - min(v)) / np.median(v)) for k, v in samples.items()}}
        row["us_per_row_host"] = row["ms"]["host"] * 1e3 / n
        row["speedup_device_copies_vs_host"] = row["ms"]["host"] / row["ms"]["device_copies"]
        rows.append(row)
        print(json.dumps(row), flush=True)

    subs = W.csv_submissions(num_images=50, objects_per_image=2500, seed=0)
    n_rows = sum(s.shape[0] for s in subs)
    ens = {"before": [], "after": []}
    outs = {}
    for r in range(a.rounds + 1):  # round 0 warms both routes up and is not recorded
        for route in ("before", "after"):
            PM._grouped_nms = grouped_nms_before if route == "before" else grouped_nms_after
            try:
                ms, outs[route] = wall(lambda: PM.merge_csv_with_class(subs, 0.625))
            finally:
                PM._grouped_nms = grouped_nms_after
            if r:
                ens[route].append(ms)
    checks["ensemble"] = bool(same(outs["before"], outs["after"]))
    ensemble = {"rows": n_rows, "kept": int(outs["after"].shape[0]),
                "ms": {k: float(np.median(v)) for k, v in ens.items()},
                "spread": {k: float((max(v) - min(v)) / np.median(v)) for k, v in ens.items()}}
    print(json.dumps(ensemble), flush=True)

    res = {"card": card(), "torch": torch.__version__, "rounds": a.rounds,
           "method": {"host": "time.perf_counter around one call, median over rounds",
                      "device": "median over rounds of CUDA-event time per call, back-to-back calls on a resident tensor",
                      "device_copies": "time.perf_counter around H2D + call + D2H, median over rounds",
                      "ensemble": "time.perf_counter around merge_csv_with_class(subs, 0.625), result on the host",
                      "spread": "(max - min) / median over rounds"},
           "poly2obb": rows, "ensemble": ensemble, "checks": checks}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    ok = all(checks.values())
    print(json.dumps({"card": res["card"], "checks_ok": ok}))
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
