"""jdet.data.devkits.result_merge (merge NMS part) -- python/jdet/data/devkits/result_merge.py.

`py_cpu_nms_poly_fast(dets, thresh)` keeps its name, numpy-in / list-out contract (:66-127) so that
`mergebypoly`, `tools/merge_results.py:38` and `nmsbynamedict` (:177-193) can call it unchanged; the
greedy loop and the Shapely call per candidate pair are replaced by the float64 merge predicate of the
device NMS engine.  `merge_detections` is the batched form: ALL (scene, class) groups of a result set
in one launch, per-class thresholds included.

File level (SURVEY §8(f) rank 4, :206-299): `mergesingle` / `mergebase` / `mergebase_parallel` / `mergebypoly`
read the per-class `before_nms/<Class>.txt` files (`tile_name score x1 y1 ... y4`, tile name
`<scene>__<rate>__<x>___<y>`), map tile polygons to scene coordinates on the device
(`rsdet_poly2origpoly`), run ONE merge-NMS launch over every (file, scene) group and write
`<scene> <score> <8 coords>` lines with the reference's `str(float)` formatting.
"""
import os
import re

import numpy as np
import torch

from .... import core
from ...._lib import NMS_HBB_P1_F64, NMS_MERGE, NMS_ROTATED_GE, require_cuda

# the thresh for nms when merge image (result_merge.py:24-27)
nms_threshold_0 = 0.1
nms_threshold_1 = {'Roundabout': 0.1, 'Tennis_Court': 0.1, 'Football_Field': 0.1, 'Vehicle': 0.15, 'Ship': 0.2,
                   'Airplane': 0.3, 'Intersection': 0.3, 'Bridge': 0.0001, 'Basketball_Court': 0.1, 'Baseball_Field': 0.1}


def py_cpu_nms_poly_fast(dets, thresh):
    """dets (n,9) float64 [x1..y4,score] -> python list of kept indices in descending-score order."""
    require_cuda()
    d = np.ascontiguousarray(dets, dtype=np.float64).reshape(-1, 9)
    if d.shape[0] == 0:
        return []
    t = torch.from_numpy(d).cuda()
    res = core.nms(NMS_MERGE, t[:, :8], t[:, 8], float(thresh), want_mask=False, want_sorted=False, want_score=True,
                   ws_tag="merge")
    return res.score_idx.cpu().tolist()


def py_cpu_nms_poly(dets, thresh):
    """:30-63 -- the same predicate as the `_fast` variant without the hbb prefilter (pairs whose hbbs do not
    overlap have IoU 0, which both variants suppress exactly when thresh < 0): one engine, same result."""
    return py_cpu_nms_poly_fast(dets, thresh)


def py_cpu_nms(dets, thresh):
    """:143-174 -- horizontal boxes (n,5) float64 [x1,y1,x2,y2,score], '+1' areas, survivors `ovr <= thresh`;
    returns the kept indices in descending-score order (python list).  A pair without a '+1' overlap whose '+1' areas
    sum to 0 has ovr = 0/0 = NaN and is suppressed, as in the reference; any other such pair has ovr = 0, suppressed
    only when thresh < 0."""
    require_cuda()
    d = np.ascontiguousarray(dets, dtype=np.float64).reshape(-1, 5)
    if d.shape[0] == 0:
        return []
    t = torch.from_numpy(d).cuda()
    res = core.nms(NMS_HBB_P1_F64, t[:, :4], t[:, 4], float(thresh), want_mask=False, want_sorted=False, want_score=True,
                   ws_tag="merge")
    return res.score_idx.cpu().tolist()


def py_cpu_nms_obb(dets, thresh):
    """:128-141 -- polygons -> oriented boxes (`poly2obb`: the device restatement of the reference's cv2.minAreaRect,
    bit for bit) -> `nms_rotated_cpu` (suppress IoU >= thresh) -> kept indices in ASCENDING index order
    (`jt.where(keep)[0]`)."""
    require_cuda()
    d = np.ascontiguousarray(dets, dtype=np.float64).reshape(-1, 9)
    if d.shape[0] == 0:
        return np.array([])
    t = torch.from_numpy(d).cuda()
    obb = core.poly2obb(t[:, :8]).to(torch.float32)
    sc = t[:, 8].to(torch.float32)
    res = core.nms(NMS_ROTATED_GE, obb, sc, float(thresh), want_mask=False, want_sorted=True, ws_tag="merge")
    return res.sorted_idx.cpu().numpy()


def poly2origpoly(poly, x, y, rate):
    """:196-203"""
    origpoly = []
    for i in range(int(len(poly) / 2)):
        origpoly.append(float(poly[i * 2] + x) / float(rate))
        origpoly.append(float(poly[i * 2 + 1] + y) / float(rate))
    return origpoly


def nmsbynamedict(nameboxdict, nms, thresh):
    """:177-193 (kept for API parity; one engine call per scene)."""
    nameboxnmsdict = {x: [] for x in nameboxdict}
    for imgname in nameboxdict:
        keep = nms(np.array(nameboxdict[imgname]), thresh)
        nameboxnmsdict[imgname] = [nameboxdict[imgname][index] for index in keep]
    return nameboxnmsdict


def merge_detections(polys, scores, group_ids, thresh=nms_threshold_0, group_thresh=None):
    """Batched merge NMS: polys (n,8) float64 scene coordinates, scores (n,), group_ids (n,) int -- one id
    per (scene, class) pair; `group_thresh`: optional per-group-id thresholds (len > max id).
    Returns kept indices in descending-score order (device int64 tensor when inputs are CUDA tensors,
    numpy otherwise)."""
    require_cuda()
    host = not (isinstance(polys, torch.Tensor) and polys.is_cuda)
    p = torch.as_tensor(polys, dtype=torch.float64).cuda() if host else polys.to(torch.float64)
    s = torch.as_tensor(scores, dtype=torch.float64).cuda() if host else scores.to(torch.float64)
    g = torch.as_tensor(group_ids).to(torch.int32).cuda() if host else group_ids.to(torch.int32)
    tpl = None
    if group_thresh is not None:
        tpl = torch.as_tensor(group_thresh, dtype=torch.float64).cuda()
    res = core.nms(NMS_MERGE, p, s, float(thresh), labels=g, thr_per_label=tpl, want_mask=False, want_sorted=False,
                   want_score=True, ws_tag="merge")
    keep = res.score_idx
    return keep.cpu().numpy() if host else keep


# ------------------------------------------------------------------------------------ file level
_XY = re.compile(r'__\d+___\d+')             # :224
_RATE = re.compile(r'__([\d+\.]+)__\d+___')  # :230
_INT = re.compile(r'\d+')


def custombasename(fullname):
    """dota_utils.py:25-26"""
    return os.path.basename(os.path.splitext(fullname)[0])


def GetFileFromThisRootDir(dir, ext=None):
    """dota_utils.py:29-40 (note: `extension in ext` is a substring test when ext is a str)."""
    out = []
    for root, _, files in os.walk(dir):
        for f in files:
            path = os.path.join(root, f)
            if ext is None or os.path.splitext(path)[1][1:] in ext:
                out.append(path)
    return out


def parse_tile_name(subname):
    """'<scene>__<rate>__<x>___<y>' -> (scene, x, y, rate) with the reference's regexes (:219-232)."""
    x, y = _INT.findall(_XY.findall(subname)[0])[:2]
    return subname.split('__')[0], int(x), int(y), float(_RATE.findall(subname)[0])


def read_tile_detections(fullname, ncoord=8):
    """One before_nms file -> (scene name per row, scene first-appearance order, tile polys (n,8) f64,
    per-row [x, y, rate] (n,3) f64, scores (n,) f64).  Text -> numbers only; no geometry on the host."""
    scenes, order, polys, offs, scores = [], [], [], [], []
    cache = {}
    with open(fullname, 'r') as f:
        for line in f:
            sp = line.strip().split(' ')
            if len(sp) < 2 + ncoord:
                continue
            t = cache.get(sp[0])
            if t is None:
                t = cache[sp[0]] = parse_tile_name(sp[0])
            if t[0] not in order:
                order.append(t[0])
            scenes.append(t[0])
            offs.append((t[1], t[2], t[3]))
            scores.append(float(sp[1]))
            polys.append([float(v) for v in sp[2:2 + ncoord]])
    return (scenes, order, np.asarray(polys, np.float64).reshape(-1, ncoord), np.asarray(offs, np.float64).reshape(-1, 3),
            np.asarray(scores, np.float64))


def _merge_files(files, dstpath, thresholds, kind=NMS_MERGE):
    """Shared body of mergesingle / mergebase / mergebypoly / mergebyrec: all files and scenes in one NMS launch (several
    when the dump holds more rows than an engine call takes, core.nms_grouped)."""
    require_cuda()
    recs = [read_tile_detections(f, 4 if kind == NMS_HBB_P1_F64 else 8) for f in files]
    gid_of, rows_gid, thr = {}, [], []
    for fi, (scenes, order, _, _, _) in enumerate(recs):
        for sc in order:
            gid_of[(fi, sc)] = len(thr)
            thr.append(float(thresholds[fi]))
        rows_gid.append(np.asarray([gid_of[(fi, sc)] for sc in scenes], np.int32))
    n = sum(r[2].shape[0] for r in recs)
    kept_rows = np.zeros((0,), np.int64)
    scene_polys = np.zeros((0, 8))
    if n > 0:
        polys = torch.from_numpy(np.concatenate([r[2] for r in recs])).cuda()
        offs = torch.from_numpy(np.concatenate([r[3] for r in recs])).cuda()
        scores = torch.from_numpy(np.concatenate([r[4] for r in recs])).cuda()
        if polys.shape[1] == 8:
            orig = core.poly2origpoly(polys, offs)
        else:  # (n,4) boxes: the same (p + offset) / rate map on two points
            orig = core.poly2origpoly(torch.cat([polys, polys], 1), offs)[:, :4].contiguous()
        # (file, scene) groups are independent: one launch when the rows fit an engine call, else split by group
        kept_rows = core.nms_grouped(kind, orig, scores, np.concatenate(rows_gid), nms_threshold_0,
                                     thr_per_label=torch.tensor(thr, dtype=torch.float64, device=orig.device))
        scene_polys = orig.cpu().numpy()
    all_scores = np.concatenate([r[4] for r in recs]) if n else np.zeros((0,))
    all_gids = np.concatenate(rows_gid) if n else np.zeros((0,), np.int32)
    per_gid = [[] for _ in thr]
    for r in kept_rows.tolist():  # already in descending-score order
        per_gid[all_gids[r]].append(r)
    os.makedirs(dstpath, exist_ok=True)
    for fi, f in enumerate(files):
        dstname = os.path.join(dstpath, custombasename(f) + '.txt')
        with open(dstname, 'w') as out:
            for sc in recs[fi][1]:
                for r in per_gid[gid_of[(fi, sc)]]:
                    out.write(sc + ' ' + str(float(all_scores[r])) + ' ' + ' '.join(map(str, scene_polys[r].tolist())) + '\n')


def _file_threshold(fullname, nms_threshold_type):
    return nms_threshold_0 if not nms_threshold_type else nms_threshold_1[custombasename(fullname)]


def mergebyobb(srcpath, dstpath, nms_threshold_type=0):
    """:301-315 -- oriented-box variant: per scene `py_cpu_nms_obb` (one engine call per scene, like nmsbynamedict)."""
    os.makedirs(dstpath, exist_ok=True)
    for f in GetFileFromThisRootDir(srcpath):
        scenes, order, polys, offs, scores = read_tile_detections(f)
        thr = _file_threshold(f, nms_threshold_type)
        orig = np.zeros((0, 8))
        if polys.shape[0]:
            orig = core.poly2origpoly(torch.from_numpy(polys).cuda(), torch.from_numpy(offs).cuda()).cpu().numpy()
        with open(os.path.join(dstpath, custombasename(f) + '.txt'), 'w') as out:
            for sc_name in order:
                rows = np.asarray([i for i, s_ in enumerate(scenes) if s_ == sc_name], np.int64)
                keep = py_cpu_nms_obb(np.concatenate([orig[rows], scores[rows, None]], 1), thr)
                for r in rows[np.asarray(keep, np.int64)]:
                    out.write(sc_name + ' ' + str(float(scores[r])) + ' ' + ' '.join(map(str, orig[r].tolist())) + '\n')


def _kind_of(nms):
    if nms is py_cpu_nms_poly_fast or nms is py_cpu_nms_poly:
        return NMS_MERGE
    if nms is py_cpu_nms:
        return NMS_HBB_P1_F64
    raise ValueError("merge: `nms` must be py_cpu_nms_poly_fast, py_cpu_nms_poly or py_cpu_nms (device predicates)")


def mergesingle(dstpath, nms, fullname, nms_threshold_type=0):
    """:206-255.  `nms` selects the device predicate (one of this module's three functions; anything else is
    rejected).  `nms_threshold_type` replaces `get_cfg()`."""
    _merge_files([fullname], dstpath, [_file_threshold(fullname, nms_threshold_type)], _kind_of(nms))


def mergebase(srcpath, dstpath, nms, nms_threshold_type=0):
    """:267-270 and mergebase_parallel :258-264 -- the 16-process pool becomes one launch."""
    files = GetFileFromThisRootDir(srcpath)
    _merge_files(files, dstpath, [_file_threshold(f, nms_threshold_type) for f in files], _kind_of(nms))


mergebase_parallel = mergebase


def mergebyrec(srcpath, dstpath, nms_threshold_type=0):
    """:273-283 -- horizontal-box result files (`tile score x1 y1 x2 y2`)."""
    mergebase(srcpath, dstpath, py_cpu_nms, nms_threshold_type)


def mergebypoly(srcpath, dstpath, nms_threshold_type=0):
    """:286-299"""
    mergebase_parallel(srcpath, dstpath, py_cpu_nms_poly_fast, nms_threshold_type)
