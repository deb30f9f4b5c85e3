#!/usr/bin/env python
"""bench.py -- headline benchmark of the rotated-box hot path (BASELINE.json configs[1]).

Workload (`config.workload`): Oriented R-CNN (orcnn_van3 config) inference hot path on synthetic
DOTA-shaped 1024x1024 tiles, 8 tiles per GPU per step, tiles sharded over ranks (weak scaling, no
data-path collective).  One tile =
    OrientedSingleRoIExtractor forward: 4000 rotated proposals, 4 FPN levels (stride 4/8/16/32, C=256,
        fp32 NCHW like Jittor), 7x7 bins, 2x2 samples  ->  (4000,256,7,7)
    obb2poly on the 4000 decoded boxes (oriented_head.py:304)
    multiclass_nms_rotated on the (4000 x 10 classes) candidates, score_thr 0.001, iou_thr 0.1,
        max_num 2000 (the per-class nms_rotated BASELINE.json names; SURVEY 3.1)
The FC head between extractor and NMS is dense GEMM in Jittor (out of scope): its outputs (class
scores, decoded boxes) are synthetic, random-init-like softmax scores.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

`value` : tiles/s, inputs resident in HBM, device-timed (CUDA events), max over ranks.  The 8 tiles of a step are a batch
          of images for the extractor (the reference's batched call, RoIs carrying their batch index): the step issues
          8 // RSDET_BENCH_ROI_BATCH extractor calls (default: ONE call for the 8 tiles) and one NMS chain per tile on a
          high-priority stream.
`e2e`   : tiles/s through the public jdet-mirror API with HOST (pinned) inputs: per tile the pyramid,
          proposals, boxes and scores are copied H2D and detections + polygons are read back D2H inside
          the timed region (copies double-buffered against compute on a second stream).
`roofline`: RoIAlignRotated forward kernel (HBM bound): the launch of the timed step (RSDET_BENCH_ROI_BATCH tiles per
          launch), timed alone (channels-last batch resident) with CUDA events recorded by the library around that kernel
          in this same process; `roofline.single_tile_launch` = the same kernel launched for one tile.
`cpu_baseline` / `--impl reference`: the reference's own kernel source compiled for the host
          (oracle/_ref; RoIAlignRotated has no CPU body in the reference, so this is its CUDA source
          run serially) on all host cores, on a bounded sample (1 tile per step).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import workloads as W  # noqa: E402

K_ROIS = 4000
NUM_CLASSES = 10
TILES_PER_GPU = 8
SCORE_THR = 0.001
IOU_THR = 0.1
MAX_NUM = 2000
EXTEND = (1.4, 1.2)
NSTREAMS = int(os.environ.get("RSDET_BENCH_STREAMS", "8"))
# tiles per extractor call in the timed step (1, 2, 4 or 8) and the priority of the NMS streams.  Measured on B200
# (profiles/README.md): larger batches amortise the persistent gather's start-up and tail (kernel fraction 0.404 / 0.433 /
# 0.447 / 0.451 for 1 / 2 / 4 / 8 tiles per call) but the gather then holds every SM for longer; with the NMS chains on
# HIGH-PRIORITY streams their CTAs are placed first whenever an SM has room, and `value` is 5 410 / 5 450 / 5 550 tiles/s for
# 2 / 4 / 8 (equal priorities: 5 195 / 5 150 / 4 860).
ROI_BATCH = int(os.environ.get("RSDET_BENCH_ROI_BATCH", "8"))
NMS_PRIO = int(os.environ.get("RSDET_BENCH_NMS_PRIO", "-1"))
assert ROI_BATCH in (1, 2, 4, 8), "RSDET_BENCH_ROI_BATCH must be 1, 2, 4 or 8"
METRIC = "tiles/s (Oriented R-CNN rotated-box hot path: RoIAlignRotated fwd + obb2poly + per-class nms_rotated)"
WORKLOAD = ("configs[1]: orcnn_van3 inference hot path, 8 synthetic 1024x1024 tiles/GPU, 4000 rotated proposals/tile, "
            "4 FPN levels C=256 fp32 NCHW, RoIAlignRotated_v1 7x7x2x2 -> obb2poly -> multiclass_nms_rotated "
            "(10 classes, score_thr 0.001, iou_thr 0.1, max 2000)")


def tile_inputs(seed):
    """numpy inputs of one tile"""
    feats = W.fpn_pyramid(1, seed)
    rois = W.proposals(K_ROIS, seed)
    boxes = W.rotated_boxes(K_ROIS, seed + 500)                      # decoded detections (synthetic head output)
    scores = W.class_scores(K_ROIS, NUM_CLASSES, seed, logit_scale=1.0)  # background = column 0
    return feats, rois, boxes, scores


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------ reference arm (CPU)
_REF_FEATS = None  # set before the worker pool forks, so the 89 MB pyramid is inherited, not pickled


def _ref_roi_chunk(args):
    from oracle import ref as R
    level, rois, scale = args
    return R.roi_fwd(_REF_FEATS[level], rois, (7, 7), scale, 2, 1, fast=True)   # -O3 build: timing, not parity


def _ref_nms_class(args):
    from oracle import ref as R
    boxes, scores, thr = args
    order = np.argsort(-scores.astype(np.float64), kind="stable").astype(np.int32)
    return R.nms_keep(boxes, order, thr, 5, ge=False, fast=True)  # the CUDA path's `>` rule; -O3 build: timing, not parity


def reference_tile(nproc, inputs):
    """One tile through the reference's own kernel source compiled for the host (oracle/_ref), all cores:
    RoIs chunked over workers per level, then one NMS task per class (= ml_nms_rotated's label gate)."""
    global _REF_FEATS
    from multiprocessing import get_context
    from oracle import oracle as O
    feats, rois, boxes, scores = inputs
    _REF_FEATS = feats
    r = O.roi_rescale(rois, EXTEND)
    lv = O.map_roi_levels(r, 4)
    tasks, slots = [], []
    for l in range(4):
        idx = np.nonzero(lv == l)[0]
        for ch in np.array_split(idx, max(1, min(4 * nproc, len(idx) // 16))):
            if len(ch):
                tasks.append((l, r[ch], 1.0 / W.STRIDES[l]))
                slots.append(ch)
    out = np.zeros((K_ROIS, W.CHANNELS, 7, 7), np.float32)
    sc = scores[:, 1:]
    ntasks = [(boxes[sc[:, c] > SCORE_THR], sc[sc[:, c] > SCORE_THR, c], IOU_THR) for c in range(NUM_CLASSES)]
    with get_context("fork").Pool(nproc) as pool:
        nms_async = pool.map_async(_ref_nms_class, ntasks, chunksize=1)
        for ch, res in zip(slots, pool.map(_ref_roi_chunk, tasks, chunksize=1)):
            out[ch] = res
        keeps = nms_async.get()
    polys = O.obb2poly(boxes)
    kept = sum(int(k.sum()) for k in keeps)
    return out, polys, kept


def run_reference(args, rank, world):
    if rank != 0:
        return
    from oracle import ref as R
    if not R.available("ref_roi_v1"):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (needs /root/reference at build time)"}))
        return
    nproc = os.cpu_count() or 1
    # the worker processes are forked and terminated; load the reference libraries in the parent as well so that the
    # driver's loaded-library record of this process shows what actually ran
    for name in ("ref_roi_v1_fast", "ref_nms5_fast", "ref_roi_v1", "ref_nms5"):
        if R.available(name):
            R._lib(name)
    inputs = tile_inputs(0)
    for _ in range(args.warmup_ref):
        reference_tile(nproc, inputs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        reference_tile(nproc, inputs)
    dt = time.perf_counter() - t0
    v = args.steps / dt
    sample = f"1 tile per step (the GPU arm runs {TILES_PER_GPU}/GPU), {args.steps} steps, {nproc} worker processes"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "tiles/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup_ref, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tiles_per_gpu": TILES_PER_GPU, "rois_per_tile": K_ROIS,
                       "nms_candidates_per_tile": K_ROIS * NUM_CLASSES, "tiles_per_step_this_arm": 1,
                       "build": "reference kernel source, g++ -O3 -march=x86-64-v3 (oracle/build_ref.py `_fast`)"},
            "cpu_baseline": {"value": v, "unit": "tiles/s", "cores": nproc, "kind": "reference", "sample": sample},
            "e2e": {"value": v, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ our arm
def touched_pixels(rois):
    """U = number of distinct feature pixels the sampling grids touch (SURVEY 8d), numpy restatement of the
    kernel's geometry; only used to size the algorithmic bytes of the roofline."""
    from oracle import oracle as O
    r = O.roi_rescale(rois, EXTEND)
    lv = O.map_roi_levels(r, 4)
    total = 0
    for l, s in enumerate(W.STRIDES):
        rr = r[lv == l]
        if not len(rr):
            continue
        H = Wd = W.TILE // s
        sc = np.float32(1.0 / s)
        cx, cy = rr[:, 1] * sc - 0.5, rr[:, 2] * sc - 0.5
        rw, rh = np.maximum(rr[:, 3] * sc, 1), np.maximum(rr[:, 4] * sc, 1)
        g = (np.arange(14) + 0.5) / 14.0 - 0.5
        xx = rw[:, None, None] * g[None, None, :]
        yy = rh[:, None, None] * g[None, :, None]
        c, sn = np.cos(rr[:, 5])[:, None, None], np.sin(rr[:, 5])[:, None, None]
        x = xx * c + yy * sn + cx[:, None, None]
        y = yy * c - xx * sn + cy[:, None, None]
        ok = (y >= -1) & (y <= H) & (x >= -1) & (x <= Wd)
        x0 = np.clip(np.floor(np.maximum(x, 0)), 0, Wd - 1).astype(np.int64)
        y0 = np.clip(np.floor(np.maximum(y, 0)), 0, H - 1).astype(np.int64)
        x1, y1 = np.minimum(x0 + 1, Wd - 1), np.minimum(y0 + 1, H - 1)
        m = np.zeros(H * Wd, bool)
        for yy_, xx_ in ((y0, x0), (y0, x1), (y1, x0), (y1, x1)):
            m[(yy_ * Wd + xx_)[ok]] = True
        total += int(m.sum())
    return total


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank to the CPUs next to its GPU (`nvidia-smi topo -m`, column "CPU Affinity") before any pinned host
    memory is allocated, so that the e2e leg's 716 MB/step of uploads come from the GPU's own NUMA node when
    several ranks share the host.  Best effort: silently keeps the inherited affinity if anything is missing."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        hdr = next(l for l in out.splitlines() if "CPU Affinity" in l)
        col = [c.strip() for c in hdr.replace("\x1b[4m", "").replace("\x1b[0m", "").split("\t")]
        row = next(l for l in out.splitlines() if l.replace("\x1b[4m", "").startswith(f"GPU{local_rank}\t") or
                   l.replace("\x1b[4m", "").startswith(f"GPU{local_rank} "))
        cells = [c.strip() for c in row.replace("\x1b[0m", "").split("\t")]
        aff = cells[col.index("CPU Affinity")]
        cpus = set()
        for part in aff.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return aff
    except Exception:
        pass
    return None


MERGE_SCENES = (("scene_90k", 20000), ("scene_250k", 55000))   # (name, true objects in the 10k x 10k scene)


def merge_component(dev, rank, world, dist, max_over_ranks, barrier):
    """BASELINE config 5 under the driver: the same synthetic 10k x 10k scene on every rank (504 tiles at rates
    0.5/1.0/1.5 emit ~4.5 near-duplicates per object), merged by `merge_sharded` -- classes over the ranks, per-class
    thresholds, one all-gather of the survivors.  Device-timed (best of 5 after 2 warm-ups), max over ranks; rank 0
    also checks the result against the unsharded single-launch engine call.  Returns a dict per scene size."""
    import torch
    from rs_detection_b200.jdet.data.devkits.result_merge import merge_detections, nms_threshold_1
    from rs_detection_b200.merge import merge_sharded, plan_class_shards
    thr = [nms_threshold_1[c] for c in W.FAIR1M_CLASSES]
    out = {}
    for name, nobj in MERGE_SCENES:
        sc = W.merge_scene(num_objects=nobj, scene=10000, seed=1)
        counts = np.bincount(sc["labels"], minlength=len(thr)).tolist()   # host knowledge: one before_nms file per class
        p, s_, l = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in (sc["polys"], sc["scores"], sc["labels"])]
        run = lambda: merge_sharded(p, s_, l, class_thr=thr, class_counts=counts)
        for _ in range(2):
            res = run()
        barrier()
        best = 1e30
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = run()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        ms = max_over_ranks(best)
        entry = {"detections": int(p.shape[0]), "n_gpus": world, "ms": ms, "boxes_per_s": p.shape[0] / (ms * 1e-3),
                 "collectives_per_call": 1 if world > 1 else 0, "owner": plan_class_shards(counts, world)}
        if rank == 0:
            kept = res.indices()
            ref = merge_detections(p, s_, l, group_thresh=thr)   # all classes in one launch on this GPU
            entry["kept"] = int(kept.numel())
            entry["matches_unsharded"] = bool(sorted(ref.tolist()) == sorted(kept.tolist()))
        out[name] = entry
        del p, s_, l
        torch.cuda.empty_cache()
    return out


def verify_tile0(tile_np, tile_dev, out_bufs, device_step, cfg, core, last_np=None):
    """Compare what one more (untimed) device step leaves behind for tile 0 with the CPU oracle: the kept set of
    `multiclass_nms_rotated` (4000 x 10 candidates, score_thr 0.001) must be identical, RoI features of 64 RoIs
    must agree to 1e-5 (relative to the tensor's scale, the contract of tests/test_gpu_roi_align.py).  The step
    extracts all tiles in one batched call: 32 RoIs of the LAST tile (batch index 7) are checked as well."""
    import torch
    from oracle import oracle as O
    feats, rois, boxes, scores = tile_np
    device_step()
    torch.cuda.synchronize()
    got_feat = out_bufs[0]                                   # tile 0's rows of the batched output
    sub = np.sort(np.random.default_rng(0).choice(K_ROIS, 64, replace=False))
    want, _ = O.oriented_extractor_fwd(feats, rois[sub], list(W.STRIDES), extend_factor=EXTEND)
    g = got_feat[torch.from_numpy(sub).to(got_feat.device)].cpu().numpy()
    scale = float(np.abs(want).max())
    roi_err = float(np.abs(g - want).max())
    if last_np is not None:
        sub2 = np.sort(np.random.default_rng(1).choice(K_ROIS, 32, replace=False))
        want2, _ = O.oriented_extractor_fwd(last_np[0], last_np[1][sub2], list(W.STRIDES), extend_factor=EXTEND)
        g2 = out_bufs[-1][torch.from_numpy(sub2).to(got_feat.device)].cpu().numpy()
        roi_err = max(roi_err, float(np.abs(g2 - want2).max()))
        scale = max(scale, float(np.abs(want2).max()))
    dets, labels, cnt = core.multiclass_nms_rotated(tile_dev[2], tile_dev[3], SCORE_THR, IOU_THR, MAX_NUM)
    k = int(cnt.item())
    wd, wl = O.multiclass_nms_rotated(boxes, scores, SCORE_THR, dict(iou_thr=IOU_THR), MAX_NUM)
    nms_ok = bool(k == wd.shape[0] and np.array_equal(dets[:k].cpu().numpy(), wd) and np.array_equal(labels[:k].cpu().numpy(), wl))
    return {"ok": bool(nms_ok and roi_err <= 1e-5 * 2 * scale), "nms_kept": k, "nms_kept_oracle": int(wd.shape[0]),
            "nms_identical": nms_ok, "roi_max_abs_err": roi_err, "roi_scale": scale,
            "roi_rois_checked": int(len(sub)) + (32 if last_np is not None else 0),
            "checksum_out_tile0": float(got_feat.double().sum())}


DUMP_ROI_ROWS = 1024   # RoI feature rows dumped (256 x 7 x 7 float32 = 50 kB each; all 32 000 would be 1.6 GB)


def dump_outputs(path, out8, step_results):
    """What the last timed step computed, as a caller of it receives it, written to path/<name>.npy (float32, or
    float64 for indices and counts; 53 MB in all): a fixed seeded sample of the RoI feature rows of the batched
    extractor output, every tile's obb2poly polygons, and every tile's kept detections and labels, concatenated in
    tile order with the per-tile counts."""
    import torch
    os.makedirs(path, exist_ok=True)
    rows = np.sort(np.random.default_rng(0).choice(out8.shape[0], DUMP_ROI_ROWS, replace=False))
    counts = [int(r[3].item()) for r in step_results]
    arrays = {
        "roi_feature_rows": rows.astype(np.float64),
        "roi_features": out8[torch.from_numpy(rows).to(out8.device)].cpu().numpy(),
        "polygons": np.stack([r[0].cpu().numpy() for r in step_results]),
        "detections": np.concatenate([r[1][:k].cpu().numpy() for r, k in zip(step_results, counts)]),
        "labels": np.concatenate([r[2][:k].cpu().numpy() for r, k in zip(step_results, counts)]).astype(np.float32),
        "detections_per_tile": np.array(counts, np.float64),
    }
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args, rank, world, local_rank):
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    import torch
    import torch.distributed as dist
    from rs_detection_b200 import _lib, core
    from rs_detection_b200.jdet.models.roi_extractors.oriented_single_level import OrientedSingleRoIExtractor
    from rs_detection_b200.jdet.ops.bbox_transforms import obb2poly
    from rs_detection_b200.jdet.ops.nms_rotated import multiclass_nms_rotated

    _lib.load()
    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    shapes = W.fpn_shapes()
    scales = [1.0 / s for s in W.STRIDES]
    cfg = core.make_roi_cfg(shapes, scales, 7, 2, 1, EXTEND, 56.0)
    cfg_cl = core.make_roi_cfg(shapes, scales, 7, 2, 1, EXTEND, 56.0, channels_last=True)
    tiles_np = [tile_inputs(1000 * rank + t) for t in range(TILES_PER_GPU)]
    # the 8 tiles of a step are a BATCH of 8 images for the extractor (one (8, C, H, W) tensor per level, RoIs carrying their
    # batch index, as the reference's extractor takes them); a tile's own tensors are views into the batch
    feats8 = [torch.from_numpy(np.concatenate([t[0][l] for t in tiles_np], 0)).to(dev) for l in range(len(shapes))]
    tiles = [([f8[i:i + 1] for f8 in feats8], torch.from_numpy(r).to(dev), torch.from_numpy(b).to(dev),
              torch.from_numpy(s).to(dev)) for i, (fs, r, b, s) in enumerate(tiles_np)]
    rois8 = torch.cat([torch.cat([torch.full((t[1].shape[0], 1), float(i), device=dev), t[1][:, 1:]], 1)
                       for i, t in enumerate(tiles)], 0).contiguous()
    shapes8 = [(TILES_PER_GPU,) + tuple(sh[1:]) for sh in shapes]
    cfg8 = core.make_roi_cfg(shapes8, scales, 7, 2, 1, EXTEND, 56.0)
    out8 = torch.empty((TILES_PER_GPU * K_ROIS, W.CHANNELS, 7, 7), dtype=torch.float32, device=dev)
    # ROI_BATCH tiles per extractor call of the timed step (RSDET_BENCH_ROI_BATCH, default all 8)
    cfgb = core.make_roi_cfg([(ROI_BATCH,) + tuple(sh[1:]) for sh in shapes], scales, 7, 2, 1, EXTEND, 56.0)
    roisb = [torch.cat([torch.cat([torch.full((K_ROIS, 1), float(j), device=dev), tiles[g * ROI_BATCH + j][1][:, 1:]], 1)
                        for j in range(ROI_BATCH)], 0).contiguous() for g in range(TILES_PER_GPU // ROI_BATCH)]
    out_buf = torch.empty((K_ROIS, W.CHANNELS, 7, 7), dtype=torch.float32, device=dev)

    # tiles are independent: they are issued round-robin on NSTREAMS streams (each with its own scratch,
    # rs_detection_b200/_lib.py keys workspaces by stream) so that the latency-bound phases of one tile
    # (sorts, greedy scan) overlap the throughput-bound phases of the others.
    side = [torch.cuda.Stream(device=dev, priority=NMS_PRIO) for _ in range(NSTREAMS)]   # NMS chains: high priority
    side2 = [torch.cuda.Stream(device=dev) for _ in range(NSTREAMS)]
    out_bufs = [out8[i * K_ROIS:(i + 1) * K_ROIS] for i in range(TILES_PER_GPU)]   # tile i's rows of the batched output

    def device_step():
        """Issue one step; returns per tile (polygons, dets, labels, count); the RoI features land in out8."""
        main = torch.cuda.current_stream()
        for st in side + side2:
            st.wait_stream(main)
        # a tile's NMS chain (sorts -> decision matrix -> per-class scan: long, mostly latency-bound) does not depend
        # on its RoI features, so it goes on a stream of its own and is issued first: the scans (10 CTAs per tile)
        # then run beside the RoI kernels instead of forming the tail of the step
        results = []
        for i, (feats, rois, boxes, scores) in enumerate(tiles):
            with torch.cuda.stream(side[i % NSTREAMS]):
                polys = core.obb2poly(boxes)
                results.append((polys,) + core.multiclass_nms_rotated(boxes, scores, SCORE_THR, IOU_THR, MAX_NUM))
        # the RoI features of all 8 tiles: ONE extractor call (32 000 RoIs; the persistent gather pays its start-up and
        # tail once per step instead of once per tile)
        for g in range(TILES_PER_GPU // ROI_BATCH):
            with torch.cuda.stream(side2[g % NSTREAMS]):
                if ROI_BATCH == TILES_PER_GPU:
                    core.roi_align_rotated_forward(cfg8, feats8, rois8, out=out8)
                else:
                    lo, hi = g * ROI_BATCH, (g + 1) * ROI_BATCH
                    core.roi_align_rotated_forward(cfgb, [f8[lo:hi] for f8 in feats8], roisb[g], out=out8[lo * K_ROIS:hi * K_ROIS])
        for st in side + side2:
            main.wait_stream(st)
        return results

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput (`value`): the step is captured ONCE into a CUDA graph (fork/join over
    # the 4 streams included) and replayed, so the ~200 launches per step cost the host 0.07 ms instead of 1.9 ms
    for _ in range(args.warmup):
        device_step()
    torch.cuda.synchronize()
    launches0 = _lib.launch_count()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step_results = device_step()   # tensors of the graph's pool: every replay rewrites them
    launches_per_step = _lib.launch_count() - launches0
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.05)  # let nvidia-smi attach before the (short) timed region
    graph.replay()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        graph.replay()
    e1.record()
    barrier()
    launches = launches_per_step * args.steps
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    value = world * TILES_PER_GPU * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:   # before anything else writes out8
        dump_outputs(args.dump_outputs, out8, step_results)

    # ---- component timings (same tiles, same process): per-kernel CUDA events
    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    reps = max(args.steps, 3)
    ms_ext = timed(lambda: [core.roi_align_rotated_forward(cfg, f, r, out=out_buf) for f, r, _, _ in tiles], reps) / TILES_PER_GPU
    ms_nms = timed(lambda: [core.multiclass_nms_rotated(b, s, SCORE_THR, IOU_THR, MAX_NUM) for _, _, b, s in tiles], reps) / TILES_PER_GPU
    feats_cl = [[core.nchw_to_nhwc(f) for f in fs] for fs, _, _, _ in tiles]
    ms_fwd_call = timed(lambda: [core.roi_align_rotated_forward(cfg_cl, fcl, t[1], out=out_buf) for fcl, t in zip(feats_cl, tiles)],
                        reps) / TILES_PER_GPU              # geometry + order + gather kernels of a channels-last call
    # the gather kernel alone: events recorded by the library around that kernel on its own stream, the 8 distinct tiles
    # cycled (713 MB of pyramids > L2), averaged over every launch
    for fcl, t in zip(feats_cl, tiles):
        core.roi_gather_kernel_ms(cfg_cl, fcl, t[1], out_buf)
    ks = [core.roi_gather_kernel_ms(cfg_cl, fcl, t[1], out_buf) for _ in range(reps) for fcl, t in zip(feats_cl, tiles)]
    ms_fwd_kernel = float(np.mean(ks))
    # the launch of the timed step: ROI_BATCH tiles go through ONE extractor call (a batch of images, RoIs with their batch
    # index), so the persistent grid pays its start-up and tail once per ROI_BATCH tiles.  Measured like the per-tile
    # launch: channels-last batch resident, library events around the gather kernel, the step's groups cycled.
    cfgb_cl = core.make_roi_cfg([(ROI_BATCH,) + tuple(sh[1:]) for sh in shapes], scales, 7, 2, 1, EXTEND, 56.0, channels_last=True)
    groups_cl = [[torch.cat([feats_cl[g * ROI_BATCH + j][l] for j in range(ROI_BATCH)], 0).contiguous() for l in range(len(shapes))]
                 for g in range(TILES_PER_GPU // ROI_BATCH)]
    outb = out8[:ROI_BATCH * K_ROIS]
    for g, fb in enumerate(groups_cl):
        core.roi_gather_kernel_ms(cfgb_cl, fb, roisb[g], outb)
    ks8 = [core.roi_gather_kernel_ms(cfgb_cl, fb, roisb[g], outb) for _ in range(reps) for g, fb in enumerate(groups_cl)]
    ms_fwd_kernel_b8 = float(np.mean(ks8))
    ms_ext8 = timed(lambda: [core.roi_align_rotated_forward(cfgb, [f8[g * ROI_BATCH:(g + 1) * ROI_BATCH] for f8 in feats8], roisb[g],
                                                            out=outb) for g in range(TILES_PER_GPU // ROI_BATCH)], reps) / TILES_PER_GPU
    del groups_cl
    # training-side figures (config 3): fwd+bwd on 512 sampled RoIs, IoU 512x2000 + assignment
    rois512 = tiles[0][1][:512].contiguous()
    gout = torch.randn((512, W.CHANNELS, 7, 7), device=dev)
    ms_fb = timed(lambda: (core.roi_align_rotated_forward(cfg, tiles[0][0], rois512),
                           core.roi_align_rotated_backward(cfg, gout, rois512, shapes)), reps)
    # backward alone (config 3): algorithmic bytes 4*K*C*49 (gradient in) + 4*C*sum(HW) (dense gradient out) + 8*C*U
    # (read-modify-write of the touched pixels) + 24*K, SURVEY 8(d); the call also zero-fills and transposes the 89 MB
    # accumulator because the caller's layout is NCHW
    ms_bwd = timed(lambda: core.roi_align_rotated_backward(cfg, gout, rois512, shapes), reps)
    U512 = float(touched_pixels(tiles_np[0][1][:512]))
    bwd_bytes = 4.0 * 512 * W.CHANNELS * 49 + 4.0 * W.CHANNELS * sum(sh[2] * sh[3] for sh in shapes) + 8.0 * W.CHANNELS * U512 + 24.0 * 512
    # config 1 (the reference's own CPU-runnable case): 2000 proposals, 15 classes, score_thr 0.05, one tile
    rois_c1 = torch.from_numpy(W.proposals(2000, 1)).to(dev)
    boxes_c1 = torch.from_numpy(W.rotated_boxes(2000, 501)).to(dev)
    scores_c1 = torch.from_numpy(W.class_scores(2000, 15, 1, logit_scale=1.0)).to(dev)
    ms_c1_roi = timed(lambda: core.roi_align_rotated_forward(cfg, tiles[0][0], rois_c1), reps)
    ms_c1_nms = timed(lambda: core.multiclass_nms_rotated(boxes_c1, scores_c1, 0.05, IOU_THR, MAX_NUM), reps)
    # config 4 (dense single-stage candidates): unlabelled nms_rotated on 100k boxes of a 4096^2 canvas, and 20k x 20k IoU
    from rs_detection_b200._lib import NMS_ROTATED
    b100k = torch.from_numpy(W.rotated_boxes(100000, 7, canvas=4096, smin=8.0, smax=128.0)).to(dev)
    s100k = torch.from_numpy(W.distinct_scores(100000, 7)).to(dev)
    ms_nms100k = timed(lambda: core.nms(NMS_ROTATED, b100k, s100k, 0.1), 3)
    b20k = b100k[:20000].contiguous()
    ms_iou20k = timed(lambda: core.box_iou_rotated(b20k, b20k, 0), 3)
    del b100k, s100k, b20k
    gt = torch.from_numpy(W.jittered_copies(tiles_np[0][1][:, 1:], 512, 3)).to(dev)
    props = tiles[0][1][:2000, 1:].contiguous()
    ms_iou = timed(lambda: core.assign_wrt_overlaps(core.box_iou_rotated(gt, props, 1, True), 0.5, 0.5, 0.5, False), reps)
    del feats_cl
    # SURVEY 8(f) rank 1: fused head tail (softmax + delta decode + threshold + obb2poly + compaction), 4000 RoIs
    gen = torch.Generator(device=dev).manual_seed(1)
    cls_logits = torch.randn((K_ROIS, NUM_CLASSES + 1), device=dev, generator=gen) * 2.0
    deltas = torch.randn((K_ROIS, 5), device=dev, generator=gen) * 0.5
    rois5 = tiles[0][1][:, 1:].contiguous()
    ms_head = timed(lambda: core.oriented_head_results(rois5, cls_logits, deltas, NUM_CLASSES, True, [0.] * 5,
                                                       [0.1, 0.1, 0.2, 0.2, 0.1], SCORE_THR, 1.0), reps)

    # SURVEY 8(f) rank 2: oriented RPN proposal stage for one 1024^2 tile (5 levels, 3 anchors, 262k anchors -> 4000)
    from rs_detection_b200.jdet.models.boxes.anchor_generator import AnchorGenerator
    rpn_shapes = [(256, 256), (128, 128), (64, 64), (32, 32), (16, 16)]
    rpn_cls_np, rpn_reg_np = W.rpn_outputs(rpn_shapes, 3, 5)
    rpn_cls = [torch.from_numpy(x).to(dev) for x in rpn_cls_np]
    rpn_reg = [torch.from_numpy(x).to(dev) for x in rpn_reg_np]
    rpn_anc = AnchorGenerator(strides=[4, 8, 16, 32, 64], ratios=[0.5, 1.0, 2.0], scales=[8]).grid_anchors(rpn_shapes, device=dev)
    ms_rpn = timed(lambda: core.rpn_proposals(rpn_cls, rpn_reg, rpn_anc, 3, True, K_ROIS, K_ROIS, 0.8, 0), reps)
    del rpn_cls, rpn_reg

    # ---- roofline of the dominant HBM kernel: roi_align_fwd_kernel (one launch per tile)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    U = float(np.mean([touched_pixels(t[1]) for t in tiles_np[:2]]))
    algo_bytes = 4.0 * K_ROIS * W.CHANNELS * 49 + 24.0 * K_ROIS + 4.0 * W.CHANNELS * U
    algo_bytes8 = ROI_BATCH * algo_bytes
    achieved = algo_bytes8 / (ms_fwd_kernel_b8 * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "roi_align_fwd77p_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "units_per_launch": f"{ROI_BATCH} tiles = {ROI_BATCH * K_ROIS} RoIs (one extractor call of the timed step)",
                "algorithmic_bytes_per_launch": algo_bytes8, "launch_ms": ms_fwd_kernel_b8, "launches_timed": len(ks8),
                "touched_pixels_per_tile": U,
                "single_tile_launch": {"launch_ms": ms_fwd_kernel, "algorithmic_bytes": algo_bytes,
                                       "frac": algo_bytes / (ms_fwd_kernel * 1e-3) / 1e9 / peak, "launches_timed": len(ks),
                                       "call_ms_with_prologue": ms_fwd_call,
                                       "note": "the same kernel launched for ONE tile (4000 RoIs): start-up and tail of the "
                                               "persistent grid are then paid per tile"}}
    prof = os.path.join(ROOT, "profiles", "roi_fwd_traffic.json")
    if os.path.exists(prof):
        try:
            if ROI_BATCH == 8:      # the committed ncu capture is of the default launch (8 tiles)
                roofline["traffic"] = float(json.load(open(prof))["dram_bytes_per_launch"])
        except Exception:
            pass

    # ---- end-to-end through the public API with host buffers
    ext = OrientedSingleRoIExtractor(dict(type='ROIAlignRotated_v1', output_size=7, sampling_ratio=2), W.CHANNELS,
                                     list(W.STRIDES), extend_factor=EXTEND)
    # one pinned slab per tile (pyramid levels, rois, boxes, scores back to back) and one device slab per slot:
    # a tile goes up as ONE 89.7 MB copy (seven separate copies cost 8 % of the box's 55 GB/s pinned H2D rate)
    def carve(flat, shapes_):
        out, off = [], 0
        for sh in shapes_:
            n = int(np.prod(sh))
            out.append(flat[off:off + n].view(sh))
            off += n
        return out

    part_shapes = [tuple(sh) for sh in shapes] + [(K_ROIS, 6), (K_ROIS, 5), (K_ROIS, NUM_CLASSES + 1)]
    slab_elems = sum(int(np.prod(sh)) for sh in part_shapes)
    pinned = []
    for fs, r, b, s_ in tiles_np:
        flat = torch.empty(slab_elems, dtype=torch.float32).pin_memory()
        for dst, src in zip(carve(flat, part_shapes), list(fs) + [r, b, s_]):
            dst.copy_(torch.from_numpy(src))
        pinned.append(flat)
    h2d_bytes = sum(f.numel() * 4 for f in pinned)
    copy_stream = torch.cuda.Stream(device=dev)
    slabs = [torch.empty(slab_elems, dtype=torch.float32, device=dev) for _ in range(2)]
    slots = []
    for sl in slabs:
        v = carve(sl, part_shapes)
        slots.append((v[:len(shapes)], v[len(shapes)], v[len(shapes) + 1], v[len(shapes) + 2]))
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    d2h = [0]

    prefetched = [False]

    def e2e_step():
        comp = torch.cuda.current_stream()
        if not prefetched[0]:
            for e in freed:
                e.record(comp)
        results = []

        def upload(i):
            sl = slots[i % 2]
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[i % 2])
                slabs[i % 2].copy_(pinned[i], non_blocking=True)
                ready[i % 2].record(copy_stream)

        if not prefetched[0]:
            upload(0)
        prefetched[0] = False
        nbytes = 0
        for i in range(TILES_PER_GPU):
            if i + 1 < TILES_PER_GPU:
                upload(i + 1)
            sl = slots[i % 2]
            comp.wait_event(ready[i % 2])
            feats_roi = ext(sl[0], sl[1])
            polys = obb2poly(sl[2])
            dets, labels = multiclass_nms_rotated(sl[2], sl[3], SCORE_THR, dict(type='nms_rotated', iou_thr=IOU_THR), MAX_NUM)
            freed[i % 2].record(comp)
            if i + 1 == TILES_PER_GPU and TILES_PER_GPU % 2 == 0:
                # steady-state serving: the next step's first tile starts its upload while this step's last tile is
                # computed and read back (the copy engine would otherwise idle at every step boundary)
                upload(0)
                prefetched[0] = True
            dh, lh, ph = dets.cpu(), labels.cpu(), polys.cpu()  # detections + polygons back to the host
            nbytes += dh.numel() * 4 + lh.numel() * 4 + ph.numel() * 4
            results.append((dh.shape[0], float(feats_roi[0, 0, 0, 0])))
        d2h[0] = nbytes
        return results

    for _ in range(max(1, args.warmup - 1)):
        e2e_step()
    barrier()
    prefetched[0] = False  # the first timed step uploads its own first tile: all K x 8 uploads are inside the region
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        e2e_step()
    b.record()
    barrier()
    ms_e2e = max_over_ranks(a.elapsed_time(b))
    e2e_val = world * TILES_PER_GPU * args.steps / (ms_e2e * 1e-3)

    # ---- config 5 (full-scene merge NMS) at this N: class-sharded over the ranks, ONE all-gather (rs_detection_b200/merge.py)
    merge_comp = merge_component(dev, rank, world, dist, max_over_ranks, barrier)

    # ---- self-check of what the timed region produced (rank 0): tile 0 against the CPU oracle
    verified = verify_tile0(tiles_np[0], tiles[0], out_bufs, device_step, cfg, core, tiles_np[-1]) if rank == 0 and not args.no_verify else None

    # ---- FP32-ALU roofline of the IoU / NMS components (SURVEY 8d): algorithmic FLOPs of the reference's rotated-IoU
    # algorithm per pair, counted by the instrumented CPU restatement on THESE inputs, x the pairs the reference
    # evaluates (every pair of the IoU matrix; n_c (n_c - 1) / 2 per class for NMS), / time / non-tensor FP32 peak
    fp32 = None
    if rank == 0:
        from oracle import oracle as O
        fl, pr = O.flop_census(gt.cpu().numpy()[:128], props.cpu().numpy(), 1)
        fpp_iou = fl / max(pr, 1)
        fl, pr = O.flop_census(tiles_np[0][2][:256], tiles_np[0][2], 0)
        fpp_nms = fl / max(pr, 1)
        peak = 148 * 128 * 2 * (clocks["sm_max_mhz"] if clocks and clocks.get("sm_max_mhz") else 1965.0) * 1e6 / 1e12
        nc = (tiles_np[0][3][:, 1:] > SCORE_THR).sum(0).astype(np.float64)
        nms_pairs = float((nc * (nc - 1) / 2).sum())
        iou_tf = 512 * 2000 * fpp_iou / (ms_iou * 1e-3) / 1e12
        nms_tf = nms_pairs * fpp_nms / (ms_nms * 1e-3) / 1e12
        fp32 = {"peak_tflops": peak, "peak_source": "148 SMs x 128 FP32 lanes x 2 (FMA) x max SM clock (non-tensor)",
                "flop_per_pair_iou_config3": fpp_iou, "flop_per_pair_nms_tile": fpp_nms,
                "iou_512x2000_assign": {"algorithmic_tflops": iou_tf, "fp32_frac": iou_tf / peak},
                "multiclass_nms_tile": {"pairs_reference": nms_pairs, "algorithmic_tflops": nms_tf, "fp32_frac": nms_tf / peak,
                                        "note": "pairs the reference evaluates per class; a fraction above 1 means the engine "
                                                "avoids algorithmic work (one shared decision matrix for all classes, exact filters)"}}

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import ref as R
        nproc = os.cpu_count() or 1
        if R.available("ref_roi_v1"):
            t0 = time.perf_counter()
            reference_tile(nproc, tiles_np[0])
            dt = time.perf_counter() - t0
            cpu_baseline = {"value": 1.0 / dt, "unit": "tiles/s", "cores": nproc, "kind": "reference",
                            "sample": "1 tile (4000 RoIs + 40k NMS candidates) through oracle/_ref = the reference's "
                                      "kernel source compiled for the host; RoI chunks / classes over all cores"}
        else:
            cpu_baseline = {"value": None, "unit": "tiles/s", "cores": nproc, "kind": "reference",
                            "sample": "oracle/_ref not built"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "tiles/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "tiles_per_gpu": TILES_PER_GPU, "rois_per_tile": K_ROIS,
                       "nms_candidates_per_tile": K_ROIS * NUM_CLASSES,
                       "l2_policy": "inputs larger than L2 (8 pyramids = 713 MB per GPU cycled every step)",
                       "streams": NSTREAMS + TILES_PER_GPU // ROI_BATCH, "launch": "one CUDA graph replay per step",
                       "step": f"8 per-tile NMS chains on 8 streams + {TILES_PER_GPU // ROI_BATCH} RoI-extractor calls of {ROI_BATCH} tiles each "
                               f"(a batch of {ROI_BATCH} images, {ROI_BATCH * K_ROIS} RoIs per call) on further streams; NMS streams at priority "
                               f"{NMS_PRIO}; e2e: per-tile calls, streamed",
                       "cpu_affinity": numa},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": "tiles/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h[0]),
                    "ms_per_step": ms_e2e / args.steps},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "verified": verified,
            "components": {
                "merge": merge_comp, "fp32": fp32,
                "roi_extractor_fwd_ms_per_tile": ms_ext, "roi_extractor_fwd_rois_per_s": K_ROIS / (ms_ext * 1e-3),
                "roi_fwd_kernel_ms_per_tile": ms_fwd_kernel, "roi_fwd_call_channels_last_ms_per_tile": ms_fwd_call,
                "roi_fwd_kernel_batched_ms_per_tile": ms_fwd_kernel_b8 / ROI_BATCH, "roi_extractor_fwd_batched_ms_per_tile": ms_ext8,
                "roi_tiles_per_extractor_call": ROI_BATCH,
                "multiclass_nms_ms_per_tile": ms_nms, "nms_boxes_per_s": K_ROIS * NUM_CLASSES / (ms_nms * 1e-3),
                "train_roi_fwd_bwd_512_ms": ms_fb, "train_roi_fwd_bwd_rois_per_s": 512 / (ms_fb * 1e-3),
                "train_roi_bwd_512": {"ms": ms_bwd, "algorithmic_bytes": bwd_bytes, "achieved_gbs": bwd_bytes / (ms_bwd * 1e-3) / 1e9,
                                      "hbm_frac": bwd_bytes / (ms_bwd * 1e-3) / 1e9 / roofline["peak"],
                                      "note": "whole call for an NCHW caller: zero-fill + scatter kernel + NHWC->NCHW transpose"},
                "config1_2000x15": {"roi_extractor_fwd_ms": ms_c1_roi, "multiclass_nms_ms": ms_c1_nms,
                                    "tile_ms_single_stream": ms_c1_roi + ms_c1_nms},
                "config4": {"nms_rotated_100k_canvas4096_thr0.1_ms": ms_nms100k, "nms_boxes_per_s": 1e5 / (ms_nms100k * 1e-3),
                            "box_iou_rotated_20k_x_20k_ms": ms_iou20k, "iou_pairs_per_s": 4e8 / (ms_iou20k * 1e-3),
                            "iou_fp32_frac": 4e8 * 382.6 / (ms_iou20k * 1e-3) / 1e12 / 74.44992},
                "iou_512x2000_assign_ms": ms_iou, "iou_pairs_per_s": 512 * 2000 / (ms_iou * 1e-3),
                "head_tail_4000x10_ms": ms_head, "head_tail_rois_per_s": K_ROIS / (ms_head * 1e-3),
                "rpn_proposals_262k_anchors_ms": ms_rpn, "rpn_anchors_per_s": 261888 / (ms_rpn * 1e-3)},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle check of tile 0 after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (inputs are seeded: two builds can "
                         "be compared output for output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.warmup_ref = min(args.warmup, 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
