"""Seeded synthetic inputs for the rotated-box hot path (numpy only; shared by tests/ and bench.py).

Shapes and distributions follow SURVEY.md section 8(d): 1024x1024 DOTA-shaped tiles, FPN strides
4/8/16/32 with C=256, rotated proposals with sqrt(w*h) log-uniform in [8,512], aspect ratio
log-uniform in [1/8,8], theta uniform in (-pi/2, pi/2) (`le90`), distinct scores.
"""
from __future__ import annotations

import numpy as np

TILE = 1024
STRIDES = (4, 8, 16, 32)
CHANNELS = 256


def rotated_boxes(n, seed=0, canvas=TILE, smin=8.0, smax=512.0, rmax=8.0, dtype=np.float32):
    """(n,5) [cx,cy,w,h,theta]."""
    rng = np.random.default_rng(seed)
    cx = rng.uniform(0, canvas, n)
    cy = rng.uniform(0, canvas, n)
    s = 2.0 ** rng.uniform(np.log2(smin), np.log2(smax), n)
    r = 2.0 ** rng.uniform(-np.log2(rmax), np.log2(rmax), n)
    w = s * np.sqrt(r)
    h = s / np.sqrt(r)
    th = rng.uniform(-np.pi / 2, np.pi / 2, n)
    return np.stack([cx, cy, w, h, th], 1).astype(dtype)


def jittered_copies(boxes, n, seed=1, pos_sigma=0.08, size_sigma=0.12, ang_sigma=0.15):
    """n boxes sampled (with replacement) from `boxes` and perturbed so IoU with the source spans 0..1."""
    rng = np.random.default_rng(seed)
    src = boxes[rng.integers(0, boxes.shape[0], n)].astype(np.float64)
    s = np.sqrt(src[:, 2] * src[:, 3])
    out = src.copy()
    out[:, 0] += rng.normal(0, pos_sigma, n) * s
    out[:, 1] += rng.normal(0, pos_sigma, n) * s
    out[:, 2] *= np.exp(rng.normal(0, size_sigma, n))
    out[:, 3] *= np.exp(rng.normal(0, size_sigma, n))
    out[:, 4] += rng.normal(0, ang_sigma, n)
    return out.astype(np.float32)


def proposals(k, seed=0, batch=1, canvas=TILE):
    """(k,6) rois [batch_idx,cx,cy,w,h,theta] as produced by arb2roi (oriented_head.py:263-277)."""
    b = rotated_boxes(k, seed, canvas)
    rng = np.random.default_rng(seed + 7919)
    idx = rng.integers(0, batch, k).astype(np.float32)
    return np.concatenate([idx[:, None], b], 1).astype(np.float32)


def fpn_shapes(batch=1, tile=TILE, channels=CHANNELS, strides=STRIDES):
    return [(batch, channels, tile // s, tile // s) for s in strides]


def fpn_pyramid(batch=1, seed=0, tile=TILE, channels=CHANNELS, strides=STRIDES):
    rng = np.random.default_rng(seed + 104729)
    return [rng.standard_normal(shp, dtype=np.float32) for shp in fpn_shapes(batch, tile, channels, strides)]


def distinct_scores(n, seed=0, lo=0.0, hi=1.0):
    """A random permutation of linspace(lo,hi) -> no ties (SURVEY 8d config 4)."""
    rng = np.random.default_rng(seed + 15485863)
    s = np.linspace(lo, hi, n + 2, dtype=np.float64)[1:-1]
    return rng.permutation(s).astype(np.float32)


def class_scores(k, num_classes, seed=0, logit_scale=3.0):
    """(k, num_classes+1) softmax scores, column 0 = background (nms_rotated.py:547-563)."""
    rng = np.random.default_rng(seed + 32452843)
    z = rng.standard_normal((k, num_classes + 1)) * logit_scale
    z -= z.max(1, keepdims=True)
    e = np.exp(z)
    p = (e / e.sum(1, keepdims=True)).astype(np.float32)
    # break ties deterministically (softmax of random normals is already a.s. distinct)
    return p


def obb_to_poly64(obb):
    """float64 obb2poly (bbox_transforms.py:612-623 convention) for building merge inputs."""
    o = np.asarray(obb, np.float64)
    cx, cy, w, h, t = [o[:, i] for i in range(5)]
    c, s = np.cos(t), np.sin(t)
    v1x, v1y = w / 2 * c, -w / 2 * s
    v2x, v2y = -h / 2 * s, -h / 2 * c
    return np.stack([cx + v1x + v2x, cy + v1y + v2y, cx + v1x - v2x, cy + v1y - v2y,
                     cx - v1x - v2x, cy - v1y - v2y, cx - v1x + v2x, cy - v1y + v2y], 1)


def merge_scene(num_objects=2000, num_classes=10, scene=10000, seed=0, tile=TILE, gap=200, rates=(0.5, 1.0, 1.5),
                jitter_px=1.0):
    """Detections of one large scene as the merge stage sees them (SURVEY 8d config 5).

    The scene is split at each rate into tile x tile windows with `gap` overlap (slide = tile-gap,
    ImgSplit_multi_process.py:98,271-293); every tile containing an object's centre emits a jittered,
    4-decimal-rounded copy in tile coordinates (data_merge.py:38-41) which is mapped back with
    poly2origpoly (result_merge.py:196-203).  Returns dict(polys (n,8) f64 scene coords, scores (n,) f64,
    labels (n,) int, tiles=#tiles).  Class frequencies are FAIR1M-like (a few dominant classes).
    """
    rng = np.random.default_rng(seed + 49979687)
    freq = np.array([0.08, 0.22, 0.45, 0.03, 0.05, 0.02, 0.03, 0.06, 0.03, 0.03][:num_classes], np.float64)
    freq = freq / freq.sum()
    cls = rng.choice(num_classes, num_objects, p=freq)
    obj = rotated_boxes(num_objects, seed + 11, canvas=scene, smin=8.0, smax=96.0, rmax=4.0, dtype=np.float64)
    base_score = rng.uniform(0.05, 1.0, num_objects)
    polys, scores, labels = [], [], []
    ntiles = 0
    slide = tile - gap
    for rate in rates:
        size = scene * rate
        starts = list(range(0, max(int(size) - tile, 0) + 1, slide))
        if starts[-1] + tile < size:
            starts.append(int(size) - tile)
        ntiles += len(starts) ** 2
        ob = obj.copy()
        ob[:, :4] *= rate
        for x0 in starts:
            inx = (ob[:, 0] >= x0) & (ob[:, 0] < x0 + tile)
            if not inx.any():
                continue
            for y0 in starts:
                m = inx & (ob[:, 1] >= y0) & (ob[:, 1] < y0 + tile)
                k = int(m.sum())
                if k == 0:
                    continue
                o = ob[m].copy()
                o[:, 0] += rng.normal(0, jitter_px, k) - x0
                o[:, 1] += rng.normal(0, jitter_px, k) - y0
                o[:, 2] *= np.exp(rng.normal(0, 0.03, k))
                o[:, 3] *= np.exp(rng.normal(0, 0.03, k))
                o[:, 4] += rng.normal(0, 0.02, k)
                p = np.round(obb_to_poly64(o), 4)
                p[:, 0::2] = (p[:, 0::2] + x0) / rate
                p[:, 1::2] = (p[:, 1::2] + y0) / rate
                polys.append(p)
                scores.append(np.clip(base_score[m] + rng.normal(0, 0.03, k), 1e-4, 1.0))
                labels.append(cls[m])
    polys = np.concatenate(polys)
    scores = np.concatenate(scores)
    labels = np.concatenate(labels)
    # distinct scores (argsort tie order is unspecified in the reference)
    scores = scores + np.arange(scores.size) * 1e-9
    perm = rng.permutation(scores.size)
    return dict(polys=polys[perm], scores=scores[perm], labels=labels[perm], tiles=ntiles)


FAIR1M_CLASSES = ['Airplane', 'Ship', 'Vehicle', 'Basketball_Court', 'Tennis_Court', 'Football_Field',
                  'Baseball_Field', 'Intersection', 'Roundabout', 'Bridge']


def csv_submissions(num_images=20, objects_per_image=500, scene=15000.0, seed=0):
    """Two FAIR1M CSV submissions of the same scenes as `merge.read_csv_to_numpy` returns them: (n,11) float64 rows
    [image id, 8 coords rounded to 4 decimals, score, class 1..10].  The second run sees the same objects with
    jittered corners and its own scores, so the ensemble NMS has overlapping pairs to suppress."""
    rng = np.random.default_rng(seed + 7919)
    subs = [[], []]
    for img in range(num_images):
        o = rotated_boxes(objects_per_image, seed * 1000 + img, canvas=scene, smin=8.0, smax=256.0, dtype=np.float64)
        cls = rng.integers(1, 11, objects_per_image)
        for run in range(2):
            q = o.copy()
            q[:, :2] += rng.normal(0, 2.0, (objects_per_image, 2))
            p = np.round(obb_to_poly64(q) + rng.normal(0, 0.5, (objects_per_image, 8)), 4)
            sc = np.round(rng.uniform(0.05, 1.0, objects_per_image), 4)
            subs[run].append(np.concatenate([np.full((objects_per_image, 1), img), p, sc[:, None], cls[:, None]], 1))
    return [np.concatenate(s) for s in subs]


def tile_results(num_objects=300, num_classes=10, scene=3000, num_scenes=2, seed=0, tile=TILE, gap=200, rates=(0.5, 1.0),
                 jitter_px=1.0):
    """The runner's per-tile result list `[((polys (k,8), scores (k,), labels (k,)), {"img_file": ...}), ...]` as
    data_merge.prepare_data reads it (data_merge.py:29-48): tile names `<scene>__<rate>__<x>___<y>.png`
    (ImgSplit naming parsed back by result_merge.py:219-232), polygons in TILE coordinates, float32.
    Scores are distinct at four decimals (the text format keeps four; argsort tie order is unspecified in the
    reference), so at most 9999 detections in total."""
    rng = np.random.default_rng(seed + 7151)
    out = []
    slide = tile - gap
    pool = rng.permutation(9999)[: 9999] + 1
    used = 0
    for s in range(num_scenes):
        name = "P%04d" % (s + 1)
        cls = rng.integers(0, num_classes, num_objects)
        obj = rotated_boxes(num_objects, seed + 31 * s + 5, canvas=scene, smin=8.0, smax=96.0, rmax=4.0, dtype=np.float64)
        for rate in rates:
            size = scene * rate
            starts = list(range(0, max(int(size) - tile, 0) + 1, slide))
            if starts[-1] + tile < size:
                starts.append(int(size) - tile)
            ob = obj.copy()
            ob[:, :4] *= rate
            for x0 in starts:
                for y0 in starts:
                    m = (ob[:, 0] >= x0) & (ob[:, 0] < x0 + tile) & (ob[:, 1] >= y0) & (ob[:, 1] < y0 + tile)
                    k = int(m.sum())
                    if k == 0:
                        continue
                    o = ob[m].copy()
                    o[:, 0] += rng.normal(0, jitter_px, k) - x0
                    o[:, 1] += rng.normal(0, jitter_px, k) - y0
                    o[:, 4] += rng.normal(0, 0.02, k)
                    if used + k > pool.size:
                        raise ValueError("tile_results: more than 9999 detections")
                    sc = pool[used:used + k] / 10000.0
                    used += k
                    rate_s = ("%g" % rate) if rate != int(rate) else "%.1f" % rate
                    out.append(((obb_to_poly64(o).astype(np.float32), sc.astype(np.float32), cls[m].astype(np.int64)),
                                {"img_file": "/data/images/%s__%s__%d___%d.png" % (name, rate_s, x0, y0)}))
    return out


def rpn_outputs(shapes=((256, 256), (128, 128), (64, 64), (32, 32), (16, 16)), num_anchors=3, seed=0, cls_per_anchor=1):
    """Synthetic `rpn_cls` / `rpn_reg` maps for one 1024x1024 tile (oriented_rpn_head.py:118-124): class logits
    N(-2, 2) (few confident anchors), deltas N(0, 0.4) with the two midpoint offsets N(0, 0.6)."""
    rng = np.random.default_rng(seed + 90001)
    cls, reg = [], []
    for h, w in shapes:
        cls.append(rng.normal(-2.0, 2.0, (num_anchors * cls_per_anchor, h, w)).astype(np.float32))
        r = rng.normal(0.0, 0.4, (num_anchors, 6, h, w)).astype(np.float32)
        r[:, 4:] = rng.normal(0.0, 0.6, (num_anchors, 2, h, w)).astype(np.float32)
        reg.append(r.reshape(num_anchors * 6, h, w))
    return cls, reg
