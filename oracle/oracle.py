"""numpy/ctypes front-end of the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import this module.  Nothing under `rs_detection_b200/` does.

* `rsdet_oracle.c`  -> `liborsdet_oracle.so`: C restatement of the reference arithmetic
  (parity PINNED against `oracle/_ref`, see the header of the C file; merge NMS UNPINNED
  because Shapely/GEOS is not available).
* the functions defined in Python below restate the reference's *glue* in numpy, each
  citing the reference file:line it follows (paths relative to /root/reference).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(HERE, "rsdet_oracle.c")
_SO = os.path.join(HERE, "liborsdet_oracle.so")

_f = np.float32
_pf = C.POINTER(C.c_float)
_pd = C.POINTER(C.c_double)
_pi = C.POINTER(C.c_int)
_pu8 = C.POINTER(C.c_uint8)


_SO_COUNT = os.path.join(HERE, "liborsdet_oracle_count.so")


def build(force: bool = False) -> str:
    """gcc -O2 -ffp-contract=off: IEEE single ops exactly as written (no FMA contraction).  Also builds the
    -DORC_COUNT_FLOPS variant `flop_census` loads, so that bench.py compiles nothing at run time."""
    for so, extra in ((_SO, []), (_SO_COUNT, ["-DORC_COUNT_FLOPS"])):
        if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(_SRC):
            subprocess.check_call(["gcc", "-std=c99", "-O2", "-ffp-contract=off", "-fno-fast-math", *extra, "-shared",
                                   "-fPIC", _SRC, "-o", so, "-lm"])
    return _SO


def flop_census(boxes1, boxes2, version: int = 1):
    """FLOPs the reference's rotated-IoU algorithm spends on `boxes1 x boxes2` (every pair, no early exit), counted by
    a -DORC_COUNT_FLOPS build of the same C restatement (SURVEY 8d).  Returns (flops, pairs)."""
    build()
    L = C.CDLL(_SO_COUNT)
    L.orc_flops_read.restype = C.c_ulonglong
    L.orc_pairs_read.restype = C.c_ulonglong
    L.orc_box_iou_rotated.argtypes = [_pf, C.c_int, _pf, C.c_int, C.c_int, C.c_int, _pf]
    b1, b2 = _c32(boxes1).reshape(-1, 5), _c32(boxes2).reshape(-1, 5)
    out = np.zeros((b1.shape[0], b2.shape[0]), np.float32)
    L.orc_flops_reset()
    L.orc_box_iou_rotated(_fp(b1), b1.shape[0], _fp(b2), b2.shape[0], version, 0, _fp(out))
    return int(L.orc_flops_read()), int(L.orc_pairs_read())


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        L.orc_rotated_iou_pair.restype = C.c_float
        L.orc_rotated_iou_pair.argtypes = [_pf, _pf, C.c_int, C.c_int, C.c_int]
        L.orc_box_iou_rotated.argtypes = [_pf, C.c_int, _pf, C.c_int, C.c_int, C.c_int, _pf]
        L.orc_nms_rotated.argtypes = [_pf, _pi, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, _pu8]
        L.orc_roi_align_rotated_fwd.argtypes = [_pf, _pf] + [C.c_int] * 4 + [C.c_float] + [C.c_int] * 4 + [_pf]
        L.orc_roi_align_rotated_bwd.argtypes = [_pf, _pf] + [C.c_int] * 5 + [C.c_float] + [C.c_int] * 4 + [_pf]
        L.orc_poly_iou.restype = C.c_float
        L.orc_poly_iou.argtypes = [_pf, _pf]
        L.orc_poly_iou_matrix.argtypes = [_pf, C.c_int, _pf, C.c_int, C.c_int, _pf]
        L.orc_poly_nms_sorted.argtypes = [_pf, C.c_int, C.c_float, _pu8]
        L.orc_convex_quad_intersection_area.restype = C.c_double
        L.orc_convex_quad_intersection_area.argtypes = [_pd, _pd]
        L.orc_iou_poly.restype = C.c_double
        L.orc_iou_poly.argtypes = [_pd, _pd]
        L.orc_merge_nms.restype = C.c_int
        L.orc_merge_nms.argtypes = [_pd, _pi, C.c_int, C.c_double, _pi]
        L.orc_hbb_nms.restype = C.c_int
        L.orc_hbb_nms.argtypes = [_pd, _pi, C.c_int, C.c_double, _pi]
        _lib = L
    return _lib


def _fp(a):
    return a.ctypes.data_as(_pf)


def _c32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


# ----------------------------------------------------------------------------- IoU
def box_iou_rotated(boxes1, boxes2, version: int = 0, sort_kind: int = 0):
    """jdet.ops.box_iou_rotated (python/jdet/ops/box_iou_rotated.py:502-509) for version 0,
    the kernel part of box_iou_rotated_v1 (box_iou_rotated_v1.py:507-513) for version 1.
    sort_kind 0 = reference CPU hull sort, 1 = reference CUDA hull sort."""
    b1, b2 = _c32(boxes1).reshape(-1, 5), _c32(boxes2).reshape(-1, 5)
    out = np.zeros((b1.shape[0], b2.shape[0]), np.float32)
    if out.size:
        lib().orc_box_iou_rotated(_fp(b1), b1.shape[0], _fp(b2), b2.shape[0], version, sort_kind, _fp(out))
    return out


def box_iou_rotated_v1(boxes1, boxes2, sort_kind: int = 0, literal_quirk: bool = False):
    """python/jdet/ops/box_iou_rotated_v1.py:507-524 including the tiny-box zeroing.

    The reference guard reads `boxes[:, [2,3]].min(1)[0] < 0.001`; Jittor's `min(dim)`
    returns values only, so `[0]` selects box 0's min side and the test degenerates to a
    scalar applied to ALL rows (literal_quirk=True reproduces that reading).  The default
    follows the evident intent (per-box test), which is what the CUDA path implements;
    the two agree whenever no box has a side < 1e-3 (all shipped fixtures)."""
    b1, b2 = _c32(boxes1).reshape(-1, 5), _c32(boxes2).reshape(-1, 5)
    ious = box_iou_rotated(b1, b2, 1, sort_kind)
    if b1.shape[0] and b2.shape[0]:
        s1 = b1[:, 2:4].min(1) < 0.001
        s2 = b2[:, 2:4].min(1) < 0.001
        if literal_quirk:
            s1 = np.full_like(s1, s1[0])
            s2 = np.full_like(s2, s2[0])
        ious[s1, :] = 0.0
        ious[:, s2] = 0.0
    return ious


# ----------------------------------------------------------------------------- assignment
def max_iou_assign(overlaps, pos_iou_thr=0.5, neg_iou_thr=0.5, min_pos_iou=0.5, match_low_quality=False,
                   gt_max_assign_all=True, gt_labels=None, assigned_labels_filled=0):
    """MaxIoUAssigner.assign_wrt_overlaps, python/jdet/models/boxes/assigner.py:111-170.
    overlaps (G, n) -> (assigned_gt_inds int32 (n,), max_overlaps (n,), labels or None).
    argmax ties resolve to the first maximum."""
    ov = np.asarray(overlaps, np.float32)
    G, n = ov.shape
    gt_inds = np.full((n,), -1, np.int32)
    argmax = ov.argmax(0)
    maxov = ov.max(0)
    if isinstance(neg_iou_thr, tuple):
        gt_inds[(maxov >= np.float32(neg_iou_thr[0])) & (maxov < np.float32(neg_iou_thr[1]))] = 0
    else:
        gt_inds[(maxov >= 0) & (maxov < np.float32(neg_iou_thr))] = 0
    pos = maxov >= np.float32(pos_iou_thr)
    gt_inds[pos] = argmax[pos] + 1
    if match_low_quality:
        gt_argmax = ov.argmax(1)
        gt_max = ov.max(1)
        for i in range(G):
            if gt_max[i] >= np.float32(min_pos_iou):
                if gt_max_assign_all:
                    gt_inds[ov[i] == gt_max[i]] = i + 1
                else:
                    gt_inds[gt_argmax[i]] = i + 1
    labels = None
    if gt_labels is not None:
        labels = np.full((n,), assigned_labels_filled, np.int32)
        p = gt_inds > 0
        labels[p] = np.asarray(gt_labels)[gt_inds[p] - 1]
    return gt_inds, maxov, labels


# ----------------------------------------------------------------------------- NMS
def _argsort_desc(scores):
    # descending, first occurrence first on ties (tests use distinct scores anyway)
    return np.argsort(-np.asarray(scores, np.float64), kind="stable").astype(np.int32)


def nms_rotated_keep(dets, order, thr, box_len=5, ge=False, sort_kind=0):
    """keep mask (bool, ORIGINAL index space): nms_rotated_cpu (ge=True,
    python/jdet/ops/nms_rotated.py:414-449,495-504) / nms_rotated_cuda (ge=False, :353-411,450-493)."""
    d = _c32(dets).reshape(-1, box_len)
    o = np.ascontiguousarray(order, np.int32)
    keep = np.zeros((d.shape[0],), np.uint8)
    if d.shape[0]:
        lib().orc_nms_rotated(_fp(d), o.ctypes.data_as(_pi), d.shape[0], box_len, float(thr), int(ge), sort_kind,
                              keep.ctypes.data_as(_pu8))
    return keep.astype(bool)


def nms_rotated(dets, scores, thr, ge=False):
    """python/jdet/ops/nms_rotated.py:527-538 -> kept indices ascending (jt.where(keep)[0])."""
    dets = _c32(dets)
    if dets.size == 0:
        return np.zeros((0,), np.int64)
    keep = nms_rotated_keep(dets, _argsort_desc(scores), thr, 5, ge)
    return np.nonzero(keep)[0]


def ml_nms_rotated(dets, scores, labels, thr, ge=False):
    """python/jdet/ops/nms_rotated.py:515-525."""
    d6 = np.concatenate([_c32(dets), np.asarray(labels).astype(np.float32)[:, None]], 1)
    keep = nms_rotated_keep(d6, _argsort_desc(scores), thr, 6, ge)
    return np.nonzero(keep)[0]


def multiclass_nms_rotated(multi_bboxes, multi_scores, score_thr, nms_cfg, max_num=-1, score_factors=None, ge=False):
    """python/jdet/ops/nms_rotated.py:540-596, including the `keep.size(0) > max_num`
    truncation quirk (max_num=-1 drops the last detection, :590-591)."""
    mb, ms = _c32(multi_bboxes), _c32(multi_scores)
    num_classes = ms.shape[1] - 1
    if mb.shape[1] > 5:
        bboxes = mb.reshape(ms.shape[0], -1, 5)[:, 1:]
    else:
        bboxes = np.broadcast_to(mb[:, None], (mb.shape[0], num_classes, 5))
    scores = ms[:, 1:]
    valid = scores > np.float32(score_thr)
    bboxes = bboxes[valid]
    if score_factors is not None:
        scores = scores * _c32(score_factors)[:, None]
    scores = scores[valid]
    labels = np.nonzero(valid)[1]
    if bboxes.size == 0:
        return np.zeros((0, 6), np.float32), np.zeros((0,), np.int32)
    iou_thr = dict(nms_cfg).get("iou_thr", 0.1)
    keep = ml_nms_rotated(bboxes, scores, labels, iou_thr, ge)
    bboxes, scores, labels = bboxes[keep], scores[keep], labels[keep]
    inds = _argsort_desc(scores)
    if keep.shape[0] > max_num:
        inds = inds[:max_num]
    bboxes, scores, labels = bboxes[inds], scores[inds], labels[inds]
    return np.concatenate([bboxes, scores[:, None]], 1), labels.astype(np.int32)


def poly_iou_matrix(p, q):
    """devPolyIoU (python/jdet/ops/nms_poly.py:113-133) on rows of 8 (or 9) floats."""
    p, q = _c32(p), _c32(q)
    assert p.shape[1] == q.shape[1] and p.shape[1] in (8, 9)
    out = np.zeros((p.shape[0], q.shape[0]), np.float32)
    if out.size:
        lib().orc_poly_iou_matrix(_fp(p), p.shape[0], _fp(q), q.shape[0], p.shape[1], _fp(out))
    return out


def poly_nms(boxes, thr):
    """python/jdet/ops/nms_poly.py:187-232 -> order_t[keep] (descending-score order)."""
    b = _c32(boxes).reshape(-1, 9)
    order = _argsort_desc(b[:, 8])
    bs = np.ascontiguousarray(b[order])
    keep = np.zeros((b.shape[0],), np.uint8)
    if b.shape[0]:
        lib().orc_poly_nms_sorted(_fp(bs), b.shape[0], float(thr), keep.ctypes.data_as(_pu8))
    return order[keep.astype(bool)].astype(np.int64)


def multiclass_poly_nms(bboxes, scores, labels, thr):
    """python/jdet/ops/nms_poly.py:234-245."""
    b = _c32(bboxes)
    max_coordinate = b.max() - b.min()
    offsets = np.asarray(labels).astype(np.float32) * (max_coordinate + np.float32(1))
    b_nms = b + offsets[:, None]
    keep = poly_nms(np.concatenate([b_nms, _c32(scores)[:, None]], 1), thr)
    dets = np.concatenate([b[keep], _c32(scores)[keep][:, None]], 1)
    return dets, np.asarray(labels)[keep]


# ----------------------------------------------------------------------------- transforms
def obb2poly(obb):
    """python/jdet/ops/bbox_transforms.py:612-623 (float32)."""
    o = _c32(obb)
    cx, cy, w, h, t = [o[..., i] for i in range(5)]
    Cos, Sin = np.cos(t), np.sin(t)
    v1x, v1y = w / 2 * Cos, -w / 2 * Sin
    v2x, v2y = -h / 2 * Sin, -h / 2 * Cos
    return np.stack([cx + v1x + v2x, cy + v1y + v2y, cx + v1x - v2x, cy + v1y - v2y,
                     cx - v1x - v2x, cy - v1y - v2y, cx - v1x + v2x, cy - v1y + v2y], -1).astype(np.float32)


def obb2hbb(obb):
    """python/jdet/ops/bbox_transforms.py:626-632."""
    o = _c32(obb)
    cx, cy, w, h, t = [o[..., i] for i in range(5)]
    Cos, Sin = np.cos(t), np.sin(t)
    xb = np.abs(w / 2 * Cos) + np.abs(h / 2 * Sin)
    yb = np.abs(w / 2 * Sin) + np.abs(h / 2 * Cos)
    return np.stack([cx - xb, cy - yb, cx + xb, cy + yb], -1).astype(np.float32)


def poly2hbb(polys):
    """python/jdet/ops/bbox_transforms.py:602-609."""
    p = _c32(polys)
    p = p.reshape(*p.shape[:-1], p.shape[-1] // 2, 2)
    return np.concatenate([p.min(-2), p.max(-2)], -1)


# ----------------------------------------------------------------------------- RoIAlignRotated
def roi_align_rotated_fwd(feat, rois, output_size, spatial_scale, sampling_ratio, version=1):
    """ROIAlignRotated_v1 (version=1, python/jdet/ops/roi_align_rotated_v1.py:300-326) /
    ROIAlignRotated (version=0, roi_align_rotated.py:256-283)."""
    feat, rois = _c32(feat), _c32(rois).reshape(-1, 6)
    N, Cc, H, W = feat.shape
    ph, pw = output_size
    out = np.zeros((rois.shape[0], Cc, ph, pw), np.float32)
    if out.size:
        lib().orc_roi_align_rotated_fwd(_fp(feat), _fp(rois), rois.shape[0], Cc, H, W, np.float32(spatial_scale),
                                        int(sampling_ratio), ph, pw, int(version), _fp(out))
    return out


def roi_align_rotated_bwd(grad, rois, feat_shape, spatial_scale, sampling_ratio, version=1):
    """_RotatedROIAlign_v1.grad, python/jdet/ops/roi_align_rotated_v1.py:327-351."""
    grad, rois = _c32(grad), _c32(rois).reshape(-1, 6)
    N, Cc, H, W = feat_shape
    gin = np.zeros(feat_shape, np.float32)
    lib().orc_roi_align_rotated_bwd(_fp(grad), _fp(rois), rois.shape[0], N, Cc, H, W, np.float32(spatial_scale),
                                    int(sampling_ratio), grad.shape[2], grad.shape[3], int(version), _fp(gin))
    return gin


def map_roi_levels(rois, num_levels, finest_scale=56):
    """OrientedSingleRoIExtractor.map_roi_levels, python/jdet/models/roi_extractors/oriented_single_level.py:53-71
    (float32 like the Jittor ops)."""
    r = _c32(rois)
    scale = np.sqrt(r[:, 3] * r[:, 4])
    lv = np.floor(np.log2(scale / np.float32(finest_scale) + np.float32(1e-6)))
    return np.clip(lv, 0, num_levels - 1).astype(np.int64)


def roi_rescale(rois, scale_factor):
    """oriented_single_level.py:73-89; scale_factor = (h_factor, w_factor)."""
    if scale_factor is None:
        return rois
    hs, ws = (scale_factor, scale_factor) if np.isscalar(scale_factor) else scale_factor
    r = _c32(rois).copy()
    r[:, 3] = np.float32(ws) * r[:, 3]
    r[:, 4] = np.float32(hs) * r[:, 4]
    return r


def oriented_extractor_fwd(feats, rois, featmap_strides, output_size=(7, 7), sampling_ratio=2,
                           extend_factor=(1.4, 1.2), finest_scale=56, version=1):
    """OrientedSingleRoIExtractor.execute, oriented_single_level.py:91-114.  Returns (roi_feats, levels)."""
    rois = _c32(rois).reshape(-1, 6)
    if len(feats) == 1:
        return roi_align_rotated_fwd(feats[0], rois, output_size, 1 / featmap_strides[0], sampling_ratio, version), None
    C_ = feats[0].shape[1]
    out = np.zeros((rois.shape[0], C_, output_size[0], output_size[1]), np.float32)
    rois = roi_rescale(rois, extend_factor)
    lv = map_roi_levels(rois, len(feats), finest_scale)
    for i in range(len(feats)):
        inds = lv == i
        if inds.any():
            out[inds] += roi_align_rotated_fwd(feats[i], rois[inds], output_size, 1 / featmap_strides[i],
                                               sampling_ratio, version)
    return out, lv


def oriented_extractor_bwd(grad, feats_shapes, rois, featmap_strides, sampling_ratio=2, extend_factor=(1.4, 1.2),
                           finest_scale=56, version=1):
    """Gradient of oriented_extractor_fwd w.r.t. each feature level (what Jittor autograd composes from
    the masked scatter + _RotatedROIAlign_v1.grad per level)."""
    rois = roi_rescale(_c32(rois).reshape(-1, 6), extend_factor)
    lv = map_roi_levels(rois, len(feats_shapes), finest_scale)
    grad = _c32(grad)
    outs = []
    for i, shp in enumerate(feats_shapes):
        inds = lv == i
        if inds.any():
            outs.append(roi_align_rotated_bwd(np.ascontiguousarray(grad[inds]), rois[inds], shp, 1 / featmap_strides[i],
                                              sampling_ratio, version))
        else:
            outs.append(np.zeros(shp, np.float32))
    return outs


# ----------------------------------------------------------------------------- merge stage
def iou_poly(p, q):
    """python/jdet/ops/nms_poly.py:247-252 (Shapely stand-in, float64; PARITY UNPINNED)."""
    p = np.ascontiguousarray(p, np.float64).reshape(8)
    q = np.ascontiguousarray(q, np.float64).reshape(8)
    return lib().orc_iou_poly(p.ctypes.data_as(_pd), q.ctypes.data_as(_pd))


def score_order(scores, stable_ties=False):
    """`scores.argsort()[::-1]` as the reference's merge paths write it.  numpy's default argsort is not stable
    (and since 2.0 vectorised), so the order of EQUAL scores is an artefact of the numpy build; `stable_ties`
    gives the well-defined variant `argsort(kind='stable')[::-1]` (higher index first), which is the device
    engine's tie rule for the float64 merge kinds."""
    s = np.asarray(scores)
    return np.ascontiguousarray((s.argsort(kind="stable") if stable_ties else s.argsort())[::-1], np.int32)


def py_cpu_nms_poly_fast(dets, thresh, stable_ties=False):
    """python/jdet/data/devkits/result_merge.py:66-127 -> list of kept indices in score order."""
    d = np.ascontiguousarray(dets, np.float64).reshape(-1, 9)
    n = d.shape[0]
    if n == 0:
        return []
    order = score_order(d[:, 8], stable_ties)
    keep = np.zeros((n,), np.int32)
    nk = lib().orc_merge_nms(d.ctypes.data_as(_pd), order.ctypes.data_as(_pi), n, float(thresh), keep.ctypes.data_as(_pi))
    return keep[:nk].tolist()


def hbb_nms(boxes, thresh, stable_ties=False):
    """merge.py:14-27 `nms` -> np.array of kept indices in score order."""
    b = np.ascontiguousarray(boxes, np.float64).reshape(-1, 5)
    n = b.shape[0]
    if n == 0:
        return np.array([], np.int64)
    order = score_order(b[:, 4], stable_ties)
    keep = np.zeros((n,), np.int32)
    nk = lib().orc_hbb_nms(b.ctypes.data_as(_pd), order.ctypes.data_as(_pi), n, float(thresh), keep.ctypes.data_as(_pi))
    return keep[:nk].astype(np.int64)


def poly2origpoly(poly, x, y, rate):
    """python/jdet/data/devkits/result_merge.py:196-203."""
    p = np.asarray(poly, np.float64).copy()
    p[..., 0::2] = (p[..., 0::2] + x) / float(rate)
    p[..., 1::2] = (p[..., 1::2] + y) / float(rate)
    return p


# ----------------------------------------------------------------------------- SURVEY 8(f) rank 1: head tail
def regular_theta(theta, mode='180', start=-np.pi / 2):
    """python/jdet/ops/bbox_transforms.py:501-507 (float32; `%` taken as floor-mod like numpy)."""
    cycle = np.float32(2 * np.pi if mode == '360' else np.pi)
    t = theta.astype(np.float32) - np.float32(start)
    t = np.mod(t, cycle).astype(np.float32)
    return t + np.float32(start)


def regular_obb(obb):
    """python/jdet/ops/bbox_transforms.py:509-519."""
    x, y, w, h, th = [obb[..., i] for i in range(5)]
    wide = w > h
    w_r = np.where(wide, w, h)
    h_r = np.where(wide, h, w)
    th_r = regular_theta(np.where(wide, th, th + np.float32(np.pi / 2)).astype(np.float32))
    return np.stack([x, y, w_r, h_r, th_r], -1).astype(np.float32)


def delta_xywht_decode(bboxes, pred, means, stds, wh_ratio_clip=16 / 1000):
    """OrientedDeltaXYWHTCoder.decode, python/jdet/models/boxes/coder.py:477-514.  bboxes (K,5), pred (K,5m)."""
    b, p = _c32(bboxes), _c32(pred)
    m = p.shape[1] // 5
    d = p.reshape(-1, m, 5) * np.asarray(stds, np.float32) + np.asarray(means, np.float32)
    dx, dy, dw, dh, dt = [d[..., i] for i in range(5)]
    mr = np.float32(np.abs(np.log(wh_ratio_clip)))
    dw, dh = np.clip(dw, -mr, mr), np.clip(dh, -mr, mr)
    px, py, pw, ph, pt = [b[:, i:i + 1] for i in range(5)]
    gx = dx * pw * np.cos(-pt) - dy * ph * np.sin(-pt) + px
    gy = dx * pw * np.sin(-pt) + dy * ph * np.cos(-pt) + py
    gw, gh = pw * np.exp(dw), ph * np.exp(dh)
    gt = regular_theta((dt + pt).astype(np.float32))
    out = regular_obb(np.stack([gx, gy, gw, gh, gt], -1).astype(np.float32))
    return out.reshape(p.shape[0], -1)


def oriented_head_get_bboxes(rois, cls_score, bbox_pred, scale_factor=None, means=(0., 0., 0., 0., 0.),
                             stds=(0.1, 0.1, 0.2, 0.2, 0.1), score_thresh=0.05):
    """OrientedHead.get_bboxes + get_results (start 'obb' -> end 'obb'),
    python/jdet/models/roi_heads/oriented_head.py:498-536, 279-305.  rois (K,6); returns (dets (M,9), labels (M,))."""
    s = _c32(cls_score)
    e = np.exp(s - s.max(1, keepdims=True))
    scores = (e / e.sum(1, keepdims=True)).astype(np.float32)
    bboxes = delta_xywht_decode(_c32(rois)[:, 1:], bbox_pred, means, stds)
    K = scores.shape[0]
    C_ = scores.shape[1] - 1
    if scale_factor is not None:
        sf = np.asarray([scale_factor] * 4 if np.isscalar(scale_factor) else scale_factor, np.float32)
        bb = bboxes.reshape(K, -1, 5).copy()
        bb[..., :4] = bb[..., :4] / sf
        bboxes = bb.reshape(K, -1)
    if bboxes.shape[1] > 5:
        bb = bboxes.reshape(K, -1, 5)
    else:
        bb = np.broadcast_to(bboxes[:, None], (K, C_, 5))
    sc = scores[:, :-1]
    valid = sc > np.float32(score_thresh)
    if not valid.any():
        return np.zeros((0, 9), np.float32), np.zeros((0,), np.int64)
    dets = np.concatenate([obb2poly(bb[valid]), sc[valid][:, None]], 1)
    return dets.astype(np.float32), np.nonzero(valid)[1].astype(np.int64)


# ----------------------------------------------------------------------------- SURVEY 8(f) rank 3: voc_eval
def voc_match(dets, gts, ovthresh=0.5):
    """TP/FP marking loop of voc_eval_dota, python/jdet/data/devkits/voc_eval.py:236-311, with `iou_poly`
    (Shapely stand-in, PARITY UNPINNED).  dets (nd,10) [img_id, 8 coords, confidence]."""
    dets = np.array(np.asarray(dets).tolist(), dtype=np.float64).reshape(-1, 10)
    confidence = dets[:, -1]
    d8 = dets[:, :-1]
    sorted_ind = np.argsort(-confidence)
    d8 = d8[sorted_ind]
    nd = len(d8)
    tp, fp = np.zeros(nd), np.zeros(nd)
    taken = {k: np.zeros(len(np.asarray(gts[k]["difficult"])), bool) for k in gts}
    for d, det in enumerate(d8):
        bb = det[1:].astype(float)
        ovmax, jmax = -np.inf, -1
        R = gts.get(int(det[0]))
        BBGT = np.asarray(R["box"], float).reshape(-1, 8) if R is not None else np.zeros((0, 8))
        if BBGT.size > 0:
            gx1, gy1 = BBGT[:, 0::2].min(1), BBGT[:, 1::2].min(1)
            gx2, gy2 = BBGT[:, 0::2].max(1), BBGT[:, 1::2].max(1)
            bx1, by1, bx2, by2 = bb[0::2].min(), bb[1::2].min(), bb[0::2].max(), bb[1::2].max()
            iw = np.maximum(np.minimum(gx2, bx2) - np.maximum(gx1, bx1) + 1., 0.)
            ih = np.maximum(np.minimum(gy2, by2) - np.maximum(gy1, by1) + 1., 0.)
            inters = iw * ih
            uni = (bx2 - bx1 + 1.) * (by2 - by1 + 1.) + (gx2 - gx1 + 1.) * (gy2 - gy1 + 1.) - inters
            keep = np.where(inters / uni > 0)[0]
            if len(keep) > 0:
                ov = [iou_poly(BBGT[k], bb) for k in keep]
                ovmax = np.max(ov)
                jmax = keep[int(np.argmax(ov))]
        if ovmax > ovthresh:
            if not np.asarray(R["difficult"]).astype(bool)[jmax]:
                if not taken[int(det[0])][jmax]:
                    tp[d] = 1.
                    taken[int(det[0])][jmax] = True
                else:
                    fp[d] = 1.
        else:
            fp[d] = 1.
    return tp, fp


# ----------------------------------------------------------------------------- SURVEY 8(f) rank 2: RPN proposals
def anchor_grid(featmap_size, stride, base_size=None, scales=(8,), ratios=(0.5, 1.0, 2.0)):
    """python/jdet/models/boxes/anchor_generator.py AnchorGenerator (mmdet v2 semantics, scale_major,
    center_offset 0): gen_single_level_base_anchors + single_level_grid_anchors -> (H*W*A, 4) float32
    [x1,y1,x2,y2] in (h, w, a) order."""
    base = np.float32(stride if base_size is None else base_size)
    r = np.asarray(ratios, np.float32)
    s = np.asarray(scales, np.float32)
    hr = np.sqrt(r)
    wr = (1 / hr).astype(np.float32)
    ws = (base * wr[:, None] * s[None, :]).reshape(-1)
    hs = (base * hr[:, None] * s[None, :]).reshape(-1)
    basea = np.stack([-0.5 * ws, -0.5 * hs, 0.5 * ws, 0.5 * hs], -1).astype(np.float32)
    H, W = featmap_size
    sx = (np.arange(W) * stride).astype(np.float32)
    sy = (np.arange(H) * stride).astype(np.float32)
    xx = np.tile(sx, H)
    yy = np.repeat(sy, W)
    shifts = np.stack([xx, yy, xx, yy], -1)
    return (basea[None, :, :] + shifts[:, None, :]).reshape(-1, 4).astype(np.float32)


def rectpoly2obb(polys):
    """python/jdet/ops/bbox_transforms.py:577-599 (float32)."""
    p = np.asarray(polys, np.float32)
    theta = np.arctan2(-(p[..., 3] - p[..., 1]), p[..., 2] - p[..., 0]).astype(np.float32)
    Cos, Sin = np.cos(theta), np.sin(theta)
    x = (((p[..., 0] + p[..., 2]) + p[..., 4]) + p[..., 6]) / np.float32(4)
    y = (((p[..., 1] + p[..., 3]) + p[..., 5]) + p[..., 7]) / np.float32(4)
    ux = p[..., 0::2] - x[..., None]
    uy = p[..., 1::2] - y[..., None]
    rx = ux * Cos[..., None] + uy * (-Sin)[..., None]
    ry = ux * Sin[..., None] + uy * Cos[..., None]
    w = rx.max(-1) - rx.min(-1)
    h = ry.max(-1) - ry.min(-1)
    return regular_obb(np.stack([x, y, w, h, theta], -1).astype(np.float32))


def midpoint_offset_decode(bboxes, pred, means=(0., 0., 0., 0., 0., 0.), stds=(1., 1., 1., 1., 0.5, 0.5), wh_ratio_clip=16 / 1000):
    """python/jdet/models/boxes/coder.py:383-433 MidpointOffsetCoder.decode, (n,4) anchors + (n,6) deltas -> (n,5)."""
    b = np.asarray(bboxes, np.float32)
    d = np.asarray(pred, np.float32) * np.asarray(stds, np.float32)[None] + np.asarray(means, np.float32)[None]
    dx, dy, dw, dh, da, db = [d[:, k] for k in range(6)]
    mr = np.float32(np.abs(np.log(wh_ratio_clip)))
    dw = np.clip(dw, -mr, mr)
    dh = np.clip(dh, -mr, mr)
    px = (b[:, 0] + b[:, 2]) * np.float32(0.5)
    py = (b[:, 1] + b[:, 3]) * np.float32(0.5)
    pw = b[:, 2] - b[:, 0]
    ph = b[:, 3] - b[:, 1]
    gw = pw * np.exp(dw)
    gh = ph * np.exp(dh)
    gx = px + pw * dx
    gy = py + ph * dy
    x1 = gx - gw * np.float32(0.5)
    y1 = gy - gh * np.float32(0.5)
    x2 = gx + gw * np.float32(0.5)
    y2 = gy + gh * np.float32(0.5)
    da = np.clip(da, np.float32(-0.5), np.float32(0.5))
    db = np.clip(db, np.float32(-0.5), np.float32(0.5))
    ga, _ga = gx + da * gw, gx - da * gw
    gb, _gb = gy + db * gh, gy - db * gh
    polys = np.stack([ga, y1, x2, gb, _ga, y2, x1, _gb], -1)
    center = np.stack([gx, gy] * 4, -1)
    cp = polys - center
    with np.errstate(divide="ignore", invalid="ignore"):
        diag = np.sqrt(cp[:, 0::2] * cp[:, 0::2] + cp[:, 1::2] * cp[:, 1::2])
        f = diag.max(-1, keepdims=True) / diag
        cp = cp * np.repeat(f, 2, axis=-1)
    return rectpoly2obb((cp + center).astype(np.float32))


def jt_nms(dets, thresh):
    """jt.nms (Jittor 1.3.4.7, python/jittor/misc.py `nms`; THIRD PARTY, not under /root/reference -- restated
    from its published source): dets (n,5) float32 [x1,y1,x2,y2,score]; argsort descending, greedy `candidate`
    selection with fail condition inter/(a_j + a_i - inter) > thresh, '+1' widths, float32 arithmetic and a double
    threshold literal.  Returns original indices in descending-score order.  Ties: lower index first (unpinned)."""
    d = np.asarray(dets, np.float32)
    order = np.argsort(-d[:, 4].astype(np.float64), kind="stable")
    b = d[order]
    one = np.float32(1)
    area = (b[:, 2] - b[:, 0] + one) * (b[:, 3] - b[:, 1] + one)
    alive = np.ones(len(b), bool)
    keep = []
    for i in range(len(b)):
        if not alive[i]:
            continue
        keep.append(i)
        iw = np.maximum(np.float32(0), np.minimum(b[i, 2], b[i + 1:, 2]) - np.maximum(b[i, 0], b[i + 1:, 0]) + one)
        ih = np.maximum(np.float32(0), np.minimum(b[i, 3], b[i + 1:, 3]) - np.maximum(b[i, 1], b[i + 1:, 1]) + one)
        inter = ih * iw
        with np.errstate(divide="ignore", invalid="ignore"):
            iou = inter / (area[i + 1:] + area[i] - inter)
        alive[i + 1:] &= ~(iou.astype(np.float64) > thresh)
    return order[np.asarray(keep, np.int64)]


def rpn_candidates(cls_scores, bbox_preds, mlvl_anchors, use_sigmoid=True, nms_pre=2000, min_bbox_size=0,
                   means=(0., 0., 0., 0., 0., 0.), stds=(1., 1., 1., 1., 0.5, 0.5)):
    """python/jdet/models/roi_heads/oriented_rpn_head.py:155-206: per-level scores, top nms_pre, decode, size filter.
    -> (proposals (m,5), scores (m,), level ids (m,), candidate row of each survivor (m,))"""
    props, scores, ids = [], [], []
    for idx, (cs, bp, anchors) in enumerate(zip(cls_scores, bbox_preds, mlvl_anchors)):
        cs = np.asarray(cs, np.float32).transpose(1, 2, 0)
        if use_sigmoid:
            x = cs.reshape(-1)
            s = (np.float32(1) / (np.float32(1) + np.exp(-x))).astype(np.float32)
        else:
            x = cs.reshape(-1, 2)
            e = np.exp(x - x.max(1, keepdims=True))
            s = (e[:, 1] / (e[:, 0] + e[:, 1])).astype(np.float32)
        bp = np.asarray(bp, np.float32).transpose(1, 2, 0).reshape(-1, 6)
        anchors = np.asarray(anchors, np.float32)
        if nms_pre > 0 and s.shape[0] > nms_pre:
            rank = np.argsort(-s.astype(np.float64), kind="stable")[:nms_pre]
            s, bp, anchors = s[rank], bp[rank], anchors[rank]
        scores.append(s)
        props.append(midpoint_offset_decode(anchors, bp, means, stds))
        ids.append(np.full(s.shape[0], idx, np.int64))
    props, scores, ids = np.concatenate(props), np.concatenate(scores), np.concatenate(ids)
    rows = np.arange(len(scores))
    if min_bbox_size >= 0:
        m = (props[:, 2] > min_bbox_size) & (props[:, 3] > min_bbox_size)
        props, scores, ids, rows = props[m], scores[m], ids[m], rows[m]
    return props, scores, ids, rows


def rpn_level_offset_nms(proposals, scores, ids, nms_thresh=0.8, nms_post=2000):
    """oriented_rpn_head.py:208-216: obb2hbb, per-level coordinate offset, jt.nms, first nms_post rows.
    -> (dets (k,6), kept rows of `proposals` in output order, offset hbbs (m,4))"""
    h = obb2hbb(proposals).astype(np.float32)
    if len(h) == 0:
        return np.zeros((0, 6), np.float32), np.zeros((0,), np.int64), h
    max_coordinate = h.max() - h.min()
    h = h + (ids.astype(np.float32) * (max_coordinate + np.float32(1)))[:, None]
    keep = jt_nms(np.concatenate([h, scores[:, None]], 1), nms_thresh)[:nms_post]
    return np.concatenate([proposals, scores[:, None]], 1)[keep], keep, h


def rpn_get_bboxes_single(cls_scores, bbox_preds, mlvl_anchors, use_sigmoid=True, nms_pre=2000, nms_post=2000, nms_thresh=0.8,
                          min_bbox_size=0, means=(0., 0., 0., 0., 0., 0.), stds=(1., 1., 1., 1., 0.5, 0.5)):
    """oriented_rpn_head.py:136-216 end to end."""
    p, s, i, _ = rpn_candidates(cls_scores, bbox_preds, mlvl_anchors, use_sigmoid, nms_pre, min_bbox_size, means, stds)
    return rpn_level_offset_nms(p, s, i, nms_thresh, nms_post)[0]


def py_cpu_nms(dets, thresh):
    """python/jdet/data/devkits/result_merge.py:143-174: horizontal NMS, float64, '+1' areas, survivors ovr <= thresh.
    Ties: higher index first (`argsort(kind='stable')[::-1]`, see score_order)."""
    d = np.asarray(dets, np.float64).reshape(-1, 5)
    x1, y1, x2, y2, sc = d[:, 0], d[:, 1], d[:, 2], d[:, 3], d[:, 4]
    areas = (x2 - x1 + 1) * (y2 - y1 + 1)
    order = score_order(sc, True).astype(np.int64)
    keep = []
    while order.size > 0:
        i = order[0]
        keep.append(int(i))
        r = order[1:]
        w = np.maximum(0.0, np.minimum(x2[i], x2[r]) - np.maximum(x1[i], x1[r]) + 1)
        h = np.maximum(0.0, np.minimum(y2[i], y2[r]) - np.maximum(y1[i], y1[r]) + 1)
        inter = w * h
        ovr = inter / (areas[i] + areas[r] - inter)
        order = r[np.where(ovr <= thresh)[0]]
    return keep
