#!/usr/bin/env python3
"""RPN anchor assignment on one 1024^2 tile: the fused call (rsdet_assign_hbb) against the routes that store the
(G, n) overlaps matrix.

    python tools/bench_anchor_assign.py [--out profiles/anchor_assign.json] [--rounds 7]

Inputs: the tile's 261 888 anchors, AnchorGenerator(strides=[4, 8, 16, 32, 64], ratios=[0.5, 1, 2], scales=[8]), and
G in {8, 64, 512, 2048} GTs, obb2hbb of workloads.jittered_copies.  Assigner: the oriented RPN's MaxIoUAssigner(0.7,
0.3, 0.3, match_low_quality=True) with GT labels.  Routes, timed alternately in every round:
  fused         core.assign_hbb
  materialised  core.bbox_overlaps + core.assign_wrt_overlaps (the library's matrix kernels)
  torch_iou     a torch broadcast IoU + core.assign_wrt_overlaps (what a user of the mirror writes without this op)
  mask_fused    core.assign_hbb with a border `valid` mask (anchor_inside_flags, allowed border 0)
  mask_compact  anchors[valid] + core.assign_hbb on the compacted anchors, scattered back (a host sync for the gather)
Each sample is CUDA events around back-to-back calls after a warm-up of every route; medians and spreads over rounds.
The routes' outputs are compared in the same run: fused, materialised and the masked pair bit for bit; torch_iou by
value (its zero IoUs may be -0.0).  The card's name and power limit are read in the same run.  Needs a GPU.
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

import workloads as W  # noqa: E402
from bench_roi_half import card, timed  # noqa: E402
from oracle import oracle as O  # noqa: E402
from rs_detection_b200 import core  # noqa: E402
from rs_detection_b200.jdet.models.boxes.anchor_generator import AnchorGenerator  # noqa: E402

LEVELS = [(256, 256), (128, 128), (64, 64), (32, 32), (16, 16)]
GTS = [8, 64, 512, 2048]
CFG = dict(pos_iou_thr=0.7, neg_iou_thr=0.3, min_pos_iou=0.3, match_low_quality=True, gt_max_assign_all=True)


def torch_iou(gt, anc):
    """The BboxOverlaps2D formula as torch broadcasting (fp32, no +1)."""
    area_g = (gt[:, 2] - gt[:, 0]) * (gt[:, 3] - gt[:, 1])
    area_a = (anc[:, 2] - anc[:, 0]) * (anc[:, 3] - anc[:, 1])
    lt = torch.max(gt[:, None, :2], anc[None, :, :2])
    rb = torch.min(gt[:, None, 2:], anc[None, :, 2:])
    wh = (rb - lt).clamp(min=0)
    overlap = wh[..., 0] * wh[..., 1]
    union = ((area_g[:, None] + area_a[None, :]) - overlap).clamp(min=1e-6)
    return overlap / union


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "anchor_assign.json"))
    ap.add_argument("--rounds", type=int, default=7)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)

    anc = torch.cat(AnchorGenerator(strides=[4, 8, 16, 32, 64], ratios=[0.5, 1.0, 2.0], scales=[8]).grid_anchors(
        LEVELS, device=dev)).contiguous()
    n = anc.shape[0]
    valid = (anc[:, 0] >= 0) & (anc[:, 1] >= 0) & (anc[:, 2] < W.TILE) & (anc[:, 3] < W.TILE)
    kw = (CFG["pos_iou_thr"], CFG["neg_iou_thr"], CFG["min_pos_iou"], CFG["match_low_quality"], CFG["gt_max_assign_all"])

    def routes(gt, labels):
        def fused():
            return core.assign_hbb(gt, anc, *kw, labels, 0)

        def materialised():
            return core.assign_wrt_overlaps(core.bbox_overlaps(gt, anc), *kw, labels, 0)

        def with_torch_iou():
            return core.assign_wrt_overlaps(torch_iou(gt, anc), *kw, labels, 0)

        def mask_fused():
            return core.assign_hbb(gt, anc, *kw, labels, 0, valid=valid)

        def mask_compact():
            idx = valid.nonzero().reshape(-1)
            r = core.assign_hbb(gt, anc[idx].contiguous(), *kw, labels, 0)
            inds = torch.full((n,), -1, dtype=torch.int32, device=dev)
            mx = torch.zeros((n,), dtype=torch.float32, device=dev)
            lab = torch.zeros((n,), dtype=torch.int32, device=dev)
            inds[idx], mx[idx], lab[idx] = r
            return inds, mx, lab

        return {"fused": fused, "materialised": materialised, "torch_iou": with_torch_iou, "mask_fused": mask_fused,
                "mask_compact": mask_compact}

    def bits_equal(x, y):
        return (torch.equal(x[0], y[0]) and torch.equal(x[1].view(torch.int32), y[1].view(torch.int32))
                and torch.equal(x[2], y[2]))

    work, checks = {}, []
    for G in GTS:
        src = W.rotated_boxes(max(G, 16), 100 + G, canvas=W.TILE, smin=8, smax=256)
        gt = torch.from_numpy(O.obb2hbb(W.jittered_copies(src, G, 200 + G))).to(dev)
        labels = torch.from_numpy(np.random.default_rng(G).integers(1, 16, G).astype(np.int32)).to(dev)
        r = routes(gt, labels)
        out = {k: f() for k, f in r.items()}
        c = {"G": G, "positives": int((out["fused"][0] > 0).sum()),
             "fused_eq_materialised_bits": bits_equal(out["fused"], out["materialised"]),
             "fused_eq_torch_iou_values": bool(torch.equal(out["fused"][0], out["torch_iou"][0])
                                               and torch.equal(out["fused"][1], out["torch_iou"][1])
                                               and torch.equal(out["fused"][2], out["torch_iou"][2])),
             "mask_fused_eq_compact_bits": bits_equal(out["mask_fused"], out["mask_compact"]),
             "repeat_bits": bits_equal(out["fused"], r["fused"]())}
        checks.append(c)
        assert all(v for k, v in c.items() if k not in ("G", "positives")), c
        del out
        work[G] = r
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    reps = {8: 20, 64: 20, 512: 5, 2048: 3}
    for G in GTS:
        for f in work[G].values():
            f()
    torch.cuda.synchronize()
    samples = {(G, k): [] for G in GTS for k in work[G]}
    for _ in range(a.rounds):
        for G in GTS:
            for k, f in work[G].items():
                samples[(G, k)].append(timed(f, reps[G]))
    rows = []
    for G in GTS:
        row = {"G": G, "anchors": n, "valid_anchors": int(valid.sum()),
               "overlaps_matrix_bytes": G * n * 4,
               "materialised_hbm_bytes": 3 * G * n * 4,   # bbox_overlaps writes it, the row and column passes read it
               "ms": {}, "spread": {}}
        for k in work[G]:
            v = samples[(G, k)]
            row["ms"][k] = float(np.median(v))
            row["spread"][k] = float((max(v) - min(v)) / np.median(v))
        row["fused_over_materialised"] = row["ms"]["fused"] / row["ms"]["materialised"]
        row["mask_fused_over_compact"] = row["ms"]["mask_fused"] / row["ms"]["mask_compact"]
        rows.append(row)
    res = {
        "what": "RPN anchor assignment, fused (rsdet_assign_hbb) vs the overlaps-matrix routes (tools/bench_anchor_assign.py)",
        "card": card(), "torch": torch.__version__,
        "workload": {"tile": W.TILE, "anchors": n, "levels": LEVELS, "ratios": [0.5, 1, 2], "scales": [8],
                     "gts": GTS, "gt_source": "obb2hbb(workloads.jittered_copies(rotated_boxes(smin=8, smax=256)))",
                     "assigner": CFG, "mask": "anchor_inside_flags, allowed border 0"},
        "method": {"rounds": a.rounds, "reps_per_sample": reps,
                   "statistic": "median over rounds of CUDA-event time per call; each round alternates every route",
                   "spread": "(max - min) / median over rounds",
                   "cache": "anchors and GTs stay resident in L2 as in a training step; the (G, n) matrix exceeds the "
                            "126 MB L2 from G = 128"},
        "checks": checks, "results": rows,
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)
    for r in rows:
        print(f"G={r['G']:>5}: " + "  ".join(f"{k} {v:.4f} ms" for k, v in r["ms"].items()))
    print(json.dumps({"card": res["card"], "checks_ok": True}))


if __name__ == "__main__":
    main()
