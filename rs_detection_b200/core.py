"""Device-level wrappers: torch CUDA tensors in, torch CUDA tensors out, one C-ABI call each.

This is the layer the `rs_detection_b200.jdet.*` mirror modules (same names / signatures as the
reference's `jdet.*`) are written on.  Nothing here computes on the host; every function raises if
librsdet.so or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import (DTYPE_BF16, DTYPE_F16, DTYPE_F32, MAX_LEVELS, NMS_HBB, NMS_MERGE, NMS_POLY, NMS_ROTATED, NMS_ROTATED_GE,
                   ROI_NHWC_MAPS, ROI_NHWC_ROIS, RoiAlignCfg, check, load, ptr, stream_ptr, workspace)

_F64_KINDS = (NMS_MERGE, NMS_HBB, 6)  # 6 = NMS_HBB_P1_F64 (py_cpu_nms)
_ROW = {NMS_ROTATED: 5, NMS_ROTATED_GE: 5, NMS_POLY: 8, NMS_MERGE: 8, NMS_HBB: 4, 5: 4, 6: 4}  # 5 = NMS_HBB_P1 (jt.nms)


def _f32(t: torch.Tensor) -> torch.Tensor:
    if not t.is_cuda:
        raise RuntimeError("expected a CUDA tensor (no CPU fallback)")
    return t.to(torch.float32).contiguous()


# ------------------------------------------------------------------------------- transforms
def obb2poly(obb: torch.Tensor) -> torch.Tensor:
    o = _f32(obb)
    n = o.numel() // 5
    out = torch.empty(*o.shape[:-1], 8, dtype=torch.float32, device=o.device)
    check(load().rsdet_obb2poly(ptr(o), n, ptr(out), stream_ptr()), "obb2poly")
    return out


def obb2hbb(obb: torch.Tensor) -> torch.Tensor:
    o = _f32(obb)
    n = o.numel() // 5
    out = torch.empty(*o.shape[:-1], 4, dtype=torch.float32, device=o.device)
    check(load().rsdet_obb2hbb(ptr(o), n, ptr(out), stream_ptr()), "obb2hbb")
    return out


def poly2hbb(polys: torch.Tensor) -> torch.Tensor:
    p = _f32(polys)
    npts = p.shape[-1] // 2
    n = p.numel() // (npts * 2) if npts else 0
    out = torch.empty(*p.shape[:-1], 4, dtype=torch.float32, device=p.device)
    check(load().rsdet_poly2hbb(ptr(p), n, max(npts, 1), ptr(out), stream_ptr()), "poly2hbb")
    return out


def poly2origpoly(polys: torch.Tensor, offs: torch.Tensor) -> torch.Tensor:
    p = polys.to(torch.float64).contiguous()
    o = offs.to(torch.float64).contiguous()
    out = torch.empty_like(p)
    check(load().rsdet_poly2origpoly(ptr(p), ptr(o), p.shape[0], ptr(out), stream_ptr()), "poly2origpoly")
    return out


def poly2obb(polys: torch.Tensor) -> torch.Tensor:
    """(n, 8) CUDA quads -> (n, 5) fp64 [cx, cy, w, h, theta]: cv2.minAreaRect of the corners as float32 points, then
    the le90 step, bit for bit as jdet.ops.bbox_transforms.poly2obb (include/rsdet.h)."""
    if not polys.is_cuda:
        raise RuntimeError("expected a CUDA tensor (no CPU fallback)")
    p = polys.to(torch.float64).contiguous()
    if p.dim() != 2 or p.shape[1] != 8:
        raise ValueError(f"poly2obb: expected (n, 8) quads, got {tuple(p.shape)}")
    out = torch.empty((p.shape[0], 5), dtype=torch.float64, device=p.device)
    check(load().rsdet_poly2obb(ptr(p), p.shape[0], ptr(out), stream_ptr()), "poly2obb")
    return out


def iou_poly_pairs(p: torch.Tensor, q: torch.Tensor) -> torch.Tensor:
    a = p.to(torch.float64).contiguous().reshape(-1, 8)
    b = q.to(torch.float64).contiguous().reshape(-1, 8)
    assert a.shape == b.shape and a.is_cuda
    out = torch.empty((a.shape[0],), dtype=torch.float64, device=a.device)
    check(load().rsdet_iou_poly_pairs(ptr(a), ptr(b), a.shape[0], ptr(out), stream_ptr()), "iou_poly_pairs")
    return out


# ------------------------------------------------------------------------------- IoU / assignment
def box_iou_rotated(boxes1: torch.Tensor, boxes2: torch.Tensor, version: int = 0, zero_tiny: bool = False) -> torch.Tensor:
    b1, b2 = _f32(boxes1), _f32(boxes2)
    n1, n2 = b1.shape[0], b2.shape[0]
    out = torch.empty((n1, n2), dtype=torch.float32, device=b1.device)
    if n1 == 0 or n2 == 0:
        return out
    L = load()
    wsb = L.rsdet_box_iou_rotated_workspace_bytes(n1, n2)
    ws = workspace(wsb)
    check(L.rsdet_box_iou_rotated(ptr(b1), n1, ptr(b2), n2, version, int(zero_tiny), ptr(out), ptr(ws), ws.numel(),
                                  stream_ptr()), "box_iou_rotated")
    return out


def _neg_range(neg_iou_thr):
    """Negatives are neg_lo <= max_overlap < neg_hi; a scalar threshold t means (0, t)."""
    if isinstance(neg_iou_thr, (tuple, list)):
        return float(neg_iou_thr[0]), float(neg_iou_thr[1])
    return 0.0, float(neg_iou_thr)


def bbox_overlaps(bboxes1: torch.Tensor, bboxes2: torch.Tensor) -> torch.Tensor:
    """BboxOverlaps2D (mode='iou', not aligned): (n1,4) x (n2,4) [x1,y1,x2,y2] -> (n1,n2) fp32 (include/rsdet.h)."""
    b1, b2 = _f32(bboxes1), _f32(bboxes2)
    n1, n2 = b1.shape[0], b2.shape[0]
    out = torch.empty((n1, n2), dtype=torch.float32, device=b1.device)
    if n1 == 0 or n2 == 0:
        return out
    check(load().rsdet_bbox_overlaps(ptr(b1), n1, ptr(b2), n2, ptr(out), stream_ptr()), "bbox_overlaps")
    return out


def assign_hbb(gt_hbb: torch.Tensor, anchors: torch.Tensor, pos_iou_thr: float, neg_iou_thr, min_pos_iou: float = 0.0,
               match_low_quality: bool = False, gt_max_assign_all: bool = True, gt_labels: Optional[torch.Tensor] = None,
               labels_fill: int = -1, valid: Optional[torch.Tensor] = None):
    """assign_wrt_overlaps(bbox_overlaps(gt_hbb, anchors), ...) bit for bit, without the (G, n) overlaps matrix.
    `valid` (n,) bool / uint8: on valid anchors the result is that of anchors[valid]; the others get -1, +0.0 and
    `labels_fill`.  Returns (gt_inds int32, max_overlaps fp32, labels int32 or None)."""
    g, a = _f32(gt_hbb), _f32(anchors)
    G, n = g.shape[0], a.shape[0]
    if G == 0 or n == 0:
        raise ValueError("No gt or proposals")
    if g.shape[-1] != 4 or a.shape[-1] != 4:
        raise ValueError("gt_hbb and anchors must be (N, 4) [x1, y1, x2, y2]")
    m = None
    if valid is not None:
        if not valid.is_cuda or valid.numel() != n:
            raise ValueError(f"valid must be a CUDA mask of {n} anchors")
        m = valid.reshape(-1).to(torch.uint8).contiguous()
    neg_lo, neg_hi = _neg_range(neg_iou_thr)
    gt_inds = torch.empty((n,), dtype=torch.int32, device=a.device)
    max_ov = torch.empty((n,), dtype=torch.float32, device=a.device)
    labels = torch.empty((n,), dtype=torch.int32, device=a.device) if gt_labels is not None else None
    gl = gt_labels.to(torch.int32).contiguous() if gt_labels is not None else None
    L = load()
    wsb = L.rsdet_assign_hbb_workspace_bytes(G, n)
    ws = workspace(wsb) if match_low_quality else None
    check(L.rsdet_assign_hbb(ptr(g), G, ptr(a), n, ptr(m), pos_iou_thr, neg_lo, neg_hi, min_pos_iou, int(match_low_quality),
                             int(gt_max_assign_all), ptr(gl), labels_fill, ptr(gt_inds), ptr(max_ov), ptr(labels), ptr(ws),
                             0 if ws is None else ws.numel(), stream_ptr()), "assign_hbb")
    return gt_inds, max_ov, labels


def assign_wrt_overlaps(overlaps: torch.Tensor, pos_iou_thr: float, neg_iou_thr, min_pos_iou: float = 0.0,
                        match_low_quality: bool = False, gt_max_assign_all: bool = True,
                        gt_labels: Optional[torch.Tensor] = None, labels_fill: int = -1):
    ov = _f32(overlaps)
    G, n = ov.shape
    if G == 0 or n == 0:
        raise ValueError("No gt or proposals")
    neg_lo, neg_hi = _neg_range(neg_iou_thr)
    gt_inds = torch.empty((n,), dtype=torch.int32, device=ov.device)
    max_ov = torch.empty((n,), dtype=torch.float32, device=ov.device)
    labels = torch.empty((n,), dtype=torch.int32, device=ov.device) if gt_labels is not None else None
    gl = gt_labels.to(torch.int32).contiguous() if gt_labels is not None else None
    L = load()
    ws = workspace(L.rsdet_assign_workspace_bytes(G))
    check(L.rsdet_assign_wrt_overlaps(ptr(ov), G, n, pos_iou_thr, neg_lo, neg_hi, min_pos_iou, int(match_low_quality),
                                      int(gt_max_assign_all), ptr(gl), labels_fill, ptr(gt_inds), ptr(max_ov), ptr(labels),
                                      ptr(ws), ws.numel(), stream_ptr()), "assign_wrt_overlaps")
    return gt_inds, max_ov, labels


# ------------------------------------------------------------------------------- NMS
class NmsResult:
    """Device-side result of one engine call; `.count` synchronises (one 4-byte D2H copy)."""

    def __init__(self, n, keep_mask, sorted_idx, score_idx, num_keep):
        self.n = n
        self._mask, self._sorted, self._score, self._num = keep_mask, sorted_idx, score_idx, num_keep
        self._count = None

    @property
    def count(self) -> int:
        if self._count is None:
            self._count = int(self._num.item()) if self.n else 0
        return self._count

    @property
    def keep_mask(self) -> torch.Tensor:
        return self._mask.bool()

    @property
    def sorted_idx(self) -> torch.Tensor:
        return self._sorted[: self.count]

    @property
    def score_idx(self) -> torch.Tensor:
        return self._score[: self.count]

    @property
    def score_idx_padded(self) -> torch.Tensor:
        """(n,) kept indices in descending score order followed by an undefined tail; no synchronisation"""
        return self._score

    @property
    def num_keep(self) -> torch.Tensor:
        """(1,) int32 device counter; no synchronisation"""
        return self._num


def nms(kind: int, dets: torch.Tensor, scores: torch.Tensor, thr: float, labels: Optional[torch.Tensor] = None,
        thr_per_label: Optional[torch.Tensor] = None, want_mask=True, want_sorted=True, want_score=False,
        ws_tag: str = "nms") -> NmsResult:
    dt = torch.float64 if kind in _F64_KINDS else torch.float32
    if not dets.is_cuda:
        raise RuntimeError("expected CUDA tensors (no CPU fallback)")
    d = dets.to(dt).contiguous()
    s = scores.to(dt).contiguous()
    n = d.shape[0]
    dev = d.device
    assert d.numel() == n * _ROW[kind], f"dets must be (n,{_ROW[kind]})"
    mask = torch.zeros((n,), dtype=torch.uint8, device=dev) if want_mask else None
    sidx = torch.empty((n,), dtype=torch.int64, device=dev) if want_sorted else None
    cidx = torch.empty((n,), dtype=torch.int64, device=dev) if want_score else None
    num = torch.zeros((1,), dtype=torch.int32, device=dev)
    if n == 0:
        return NmsResult(0, mask, sidx, cidx, num)
    lab = labels.to(torch.int32).contiguous() if labels is not None else None
    tpl = thr_per_label.to(torch.float64).contiguous() if thr_per_label is not None else None
    L = load()
    wsb = L.rsdet_nms_workspace_bytes(kind, n)
    ws = workspace(wsb, ws_tag)
    check(L.rsdet_nms(kind, ptr(d), ptr(s), ptr(lab), n, float(thr), ptr(tpl), 0 if tpl is None else tpl.numel(), ptr(mask),
                      ptr(sidx), ptr(cidx), ptr(num), ptr(ws), ws.numel(), stream_ptr()), "nms")
    return NmsResult(n, mask, sidx, cidx, num)


MAX_NMS_ROWS = 1 << 18        # engine limit per call (include/rsdet.h)


def nms_grouped(kind: int, dets: torch.Tensor, scores: torch.Tensor, group_ids, thr: float,
                thr_per_label: Optional[torch.Tensor] = None, max_rows: int = 1 << 17, ws_tag: str = "merge") -> np.ndarray:
    """Greedy NMS inside every group for ANY number of rows: `group_ids` (host int array, one id per row; a group is a
    (file, scene) pair in the merge stage) are independent NMS problems, so when the rows exceed what one engine call
    takes (n <= 2^18, and a dense-fallback workspace that grows with n^2/8 bytes) they are split BY GROUP into several
    calls of at most `max_rows` rows each (a group larger than that goes alone).  A full FAIR1M / DOTA `before_nms`
    dump at a low score threshold has more than 2^18 rows; the reference (one NMS per file and scene) has no such limit.
    Returns the kept ORIGINAL row indices (numpy int64); rows of one group come out in descending score order."""
    g = np.ascontiguousarray(np.asarray(group_ids), dtype=np.int64)
    n = g.shape[0]
    if n == 0:
        return np.zeros((0,), np.int64)

    def one(idx_t, lab_np):
        d = dets if idx_t is None else dets[idx_t]
        sc = scores if idx_t is None else scores[idx_t]
        res = nms(kind, d, sc, thr, labels=torch.from_numpy(lab_np.astype(np.int32)).to(dets.device), thr_per_label=thr_per_label,
                  want_mask=False, want_sorted=False, want_score=True, ws_tag=ws_tag)
        return res.score_idx.cpu().numpy()

    if n <= max_rows:
        return one(None, g)
    perm = np.argsort(g, kind="stable")               # rows by group, original order inside a group (tie rule intact)
    gs = g[perm]
    starts = np.flatnonzero(np.r_[True, gs[1:] != gs[:-1]])
    ends = np.r_[starts[1:], n]
    kept, lo = [], 0
    while lo < len(starts):
        hi = lo + 1
        while hi < len(starts) and ends[hi] - starts[lo] <= max_rows:
            hi += 1
        rows = perm[starts[lo]:ends[hi - 1]]
        if rows.shape[0] > MAX_NMS_ROWS:
            raise RuntimeError(f"merge NMS: one group holds {rows.shape[0]} rows; the engine takes at most {MAX_NMS_ROWS} per group")
        k = one(torch.from_numpy(rows).to(dets.device), g[rows])
        kept.append(rows[k])
        lo = hi
    return np.concatenate(kept)


def multiclass_nms_rotated(multi_bboxes: torch.Tensor, multi_scores: torch.Tensor, score_thr: float, iou_thr: float,
                           max_num: int = -1, score_factors: Optional[torch.Tensor] = None, ws_tag: str = "nms"):
    """Returns (dets (cap,6), labels (cap,), count tensor (1,) int32) -- all on device, no sync."""
    mb, ms = _f32(multi_bboxes), _f32(multi_scores)
    n, C1 = ms.shape
    nc = C1 - 1
    cap = max(n * nc, 1)
    dev = ms.device
    out = torch.empty((cap, 6), dtype=torch.float32, device=dev)
    lab = torch.empty((cap,), dtype=torch.int32, device=dev)
    cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    if n == 0:
        return out, lab, cnt
    sf = _f32(score_factors) if score_factors is not None else None
    L = load()
    wsb = L.rsdet_multiclass_nms_rotated_workspace_bytes(n, nc)
    ws = workspace(wsb, ws_tag)
    check(L.rsdet_multiclass_nms_rotated(ptr(mb), mb.shape[1], ptr(ms), n, nc, score_thr, iou_thr, int(max_num), ptr(sf),
                                         ptr(out), ptr(lab), ptr(cnt), ptr(ws), ws.numel(), stream_ptr()),
          "multiclass_nms_rotated")
    return out, lab, cnt


# ------------------------------------------------------------------------------- RoIAlignRotated
def make_roi_cfg(feat_shapes: Sequence[Sequence[int]], spatial_scales: Sequence[float], output_size, sampling_ratio: int,
                 version: int = 1, extend=(1.0, 1.0), finest_scale: float = 56.0, channels_last: bool = False) -> RoiAlignCfg:
    """feat_shapes: logical (N,C,H,W) per level; extend = (h_factor, w_factor) like the reference's
    `extend_factor` (oriented_single_level.py:85-88)."""
    cfg = RoiAlignCfg()
    L = len(feat_shapes)
    if not 1 <= L <= MAX_LEVELS:
        raise ValueError("1..8 feature levels")
    cfg.num_levels = L
    cfg.batch, cfg.channels = int(feat_shapes[0][0]), int(feat_shapes[0][1])
    for l, shp in enumerate(feat_shapes):
        if int(shp[0]) != cfg.batch or int(shp[1]) != cfg.channels:
            raise ValueError("all levels must share batch and channels")
        cfg.height[l], cfg.width[l] = int(shp[2]), int(shp[3])
        cfg.spatial_scale[l] = float(spatial_scales[l])
    ph, pw = (output_size, output_size) if isinstance(output_size, int) else output_size
    cfg.pooled_h, cfg.pooled_w = int(ph), int(pw)
    cfg.sampling_ratio = int(sampling_ratio)
    cfg.version = int(version)
    cfg.extend_h, cfg.extend_w = float(extend[0]), float(extend[1])
    cfg.finest_scale = float(finest_scale)
    cfg.channels_last = int(channels_last)
    return cfg


def _ptr_array(tensors):
    arr = (C.c_void_p * MAX_LEVELS)()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr


# element types the RoIAlignRotated entry points read and write natively (include/rsdet.h)
_ROI_DTYPES = {torch.float32: DTYPE_F32, torch.float16: DTYPE_F16, torch.bfloat16: DTYPE_BF16}


def roi_feature_dtype(feats: Sequence[torch.Tensor]) -> torch.dtype:
    """The element type the kernels read: fp16 and bf16 levels pass through uncast (all levels must then share that
    dtype, else ValueError); any other dtype is cast to fp32."""
    dtypes = {f.dtype for f in feats}
    half = dtypes & {torch.float16, torch.bfloat16}
    if not half:
        return torch.float32
    if len(dtypes) > 1:
        raise ValueError(f"RoIAlignRotated: feature levels mix dtypes {sorted(str(d) for d in dtypes)}")
    return half.pop()


def _strictly_channels_last(t: torch.Tensor) -> bool:
    """A 4-d tensor laid out (N, H, W, C) in memory that is not also plainly contiguous (C == 1 or H * W == 1 makes the
    two layouts the same memory order; such a tensor takes the contiguous route)."""
    return t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()


def roi_maps_channels_last(feats: Sequence[torch.Tensor]) -> bool:
    """Whether every level is a channels_last (N, C, H, W) tensor of a dtype the kernels read (fp32, fp16, bf16): such
    pyramids get their gradient maps channels_last."""
    return len(feats) > 0 and all(f.dtype in _ROI_DTYPES and _strictly_channels_last(f) for f in feats)


def roi_maps_native(feats: Sequence[torch.Tensor]) -> bool:
    """Whether the forward reads the levels as they are (RSDET_ROI_NHWC_MAPS): channels_last levels whose bases meet the
    fast kernels' alignment rule of include/rsdet.h (four elements: 16 bytes fp32, 8 bytes half).  Any other base would
    run the generic kernel, whose sums differ in the last bits from the fast kernels'; such levels take the NCHW route."""
    return roi_maps_channels_last(feats) and all(f.data_ptr() % (4 * f.element_size()) == 0 for f in feats)


def _roi_cfg_with(cfg: RoiAlignCfg, bits: int) -> RoiAlignCfg:
    if not bits:
        return cfg
    c = RoiAlignCfg.from_buffer_copy(cfg)
    c.channels_last |= bits
    return c


def roi_align_rotated_forward(cfg: RoiAlignCfg, feats: Sequence[torch.Tensor], rois: torch.Tensor, want_levels: bool = False,
                              out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
                              memory_format: torch.memory_format = torch.contiguous_format):
    """Half-precision levels (fp16 / bf16) are read natively; `out_dtype` is fp32 (None) or the levels' dtype.  An fp32
    output equals, bit for bit, the call on the levels converted to fp32; a half output is that result rounded once.

    Channels_last levels (logical (N, C, H, W)) are read in place when `roi_maps_native` holds; any other levels are
    made contiguous first.  The output is a new (K, C, ph, pw) tensor in `memory_format` (torch.contiguous_format or
    torch.channels_last), or `out`, contiguous or channels_last.  Layouts never change the values."""
    fdt = roi_feature_dtype(feats)
    odt = torch.float32 if out_dtype is None else out_dtype
    if odt not in (torch.float32, fdt):
        raise ValueError(f"RoIAlignRotated: out_dtype must be float32 or the features' {fdt}, got {odt}")
    if out is not None and out.dtype != odt:
        raise ValueError(f"RoIAlignRotated: out has dtype {out.dtype}, expected {odt}")
    if memory_format not in (torch.contiguous_format, torch.channels_last):
        raise ValueError(f"RoIAlignRotated: memory_format must be torch.contiguous_format or torch.channels_last, "
                         f"got {memory_format}")
    bits = 0
    if not cfg.channels_last & ROI_NHWC_MAPS and roi_maps_native(feats):
        bits |= ROI_NHWC_MAPS
        if not all(f.is_cuda for f in feats):
            raise RuntimeError("expected a CUDA tensor (no CPU fallback)")
    elif fdt == torch.float32:
        feats = [_f32(f) for f in feats]
    elif all(f.is_cuda for f in feats):
        feats = [f.contiguous() for f in feats]
    else:
        raise RuntimeError("expected a CUDA tensor (no CPU fallback)")
    r = _f32(rois)
    if r.dim() != 2 or r.shape[1] != 6:
        raise AssertionError("rois must be (K,6)")  # roi_align_rotated_v1.py:306
    K = r.shape[0]
    dev = r.device
    if out is None:
        out = torch.empty((K, cfg.channels, cfg.pooled_h, cfg.pooled_w), dtype=odt, device=dev, memory_format=memory_format)
    if _strictly_channels_last(out):
        bits |= ROI_NHWC_ROIS
    elif not out.is_contiguous():
        raise ValueError("RoIAlignRotated: out must be contiguous or channels_last")
    cfg = _roi_cfg_with(cfg, bits)
    lv = torch.empty((K,), dtype=torch.int32, device=dev) if want_levels else None
    if K:
        L = load()
        wsb = L.rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), K, 0, _ROI_DTYPES[fdt])
        ws = workspace(wsb, "roi")
        check(L.rsdet_roi_align_rotated_forward_typed(C.byref(cfg), _ROI_DTYPES[fdt], _ptr_array(feats), ptr(r), K,
                                                      _ROI_DTYPES[odt], ptr(out), ptr(lv), ptr(ws), ws.numel(), stream_ptr()),
              "roi_align_rotated_forward")
    return (out, lv) if want_levels else out


def roi_gather_kernel_ms(cfg: RoiAlignCfg, feats: Sequence[torch.Tensor], rois: torch.Tensor, out: torch.Tensor) -> float:
    """Duration (ms) of the gather kernel alone of one forward call: CUDA events recorded by the library right before
    and after that kernel on the launching stream (`rsdet_roi_align_profile_events`).  Synchronises."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); b.record()                       # materialise the cudaEvent_t handles
    check(load().rsdet_roi_align_profile_events(C.c_void_p(a.cuda_event), C.c_void_p(b.cuda_event)), "roi_align_profile_events")
    roi_align_rotated_forward(cfg, feats, rois, out=out, out_dtype=out.dtype)
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def roi_align_rotated_backward(cfg: RoiAlignCfg, grad_out: torch.Tensor, rois: torch.Tensor, feat_shapes,
                               feat_dtype: torch.dtype = torch.float32, deterministic: bool = False,
                               memory_format: torch.memory_format = torch.contiguous_format):
    """-> gradient maps in `feat_dtype` (fp32, fp16 or bf16; accumulated in fp32, rounded once).  A grad_out in fp32 or
    in `feat_dtype` is read natively, any other dtype is cast to fp32.  A channels_last grad_out is read in place, a
    contiguous one as it is, any other is made contiguous first.  `memory_format=torch.channels_last` returns logical
    (N, C, H, W) maps laid out channels_last, written so by the library (no transpose).

    deterministic=False: the atomic backward (sums in an unspecified order).  deterministic=True: every gradient element
    is the reference's sequential fp32 sum in the reference's order, the same bits on every run
    (`rsdet_roi_align_rotated_backward_deterministic`); it needs a fixed sampling grid (sampling_ratio > 0, ValueError
    otherwise) and at most 2^28 terms K * PH * PW * sampling_ratio^2 * 4 (RuntimeError above)."""
    if feat_dtype not in _ROI_DTYPES:
        raise ValueError(f"RoIAlignRotated: gradient maps can be float32, float16 or bfloat16, not {feat_dtype}")
    if memory_format not in (torch.contiguous_format, torch.channels_last):
        raise ValueError(f"RoIAlignRotated: memory_format must be torch.contiguous_format or torch.channels_last, "
                         f"got {memory_format}")
    if not grad_out.is_cuda:
        raise RuntimeError("expected a CUDA tensor (no CPU fallback)")
    g = grad_out if grad_out.dtype in (torch.float32, feat_dtype) else grad_out.to(torch.float32)
    bits = 0
    if _strictly_channels_last(g):
        bits |= ROI_NHWC_ROIS
    else:
        g = g.contiguous()
    maps_cl = memory_format == torch.channels_last and not cfg.channels_last & ROI_NHWC_MAPS
    if maps_cl:
        bits |= ROI_NHWC_MAPS
    r = _f32(rois)
    K = r.shape[0]
    dev = r.device
    grads = []
    for l, shp in enumerate(feat_shapes):
        n, c, h, w = [int(v) for v in shp]
        if maps_cl:
            grads.append(torch.empty((n, c, h, w), dtype=feat_dtype, device=dev, memory_format=torch.channels_last))
        else:
            grads.append(torch.empty((n, h, w, c) if cfg.channels_last & ROI_NHWC_MAPS else (n, c, h, w), dtype=feat_dtype,
                                     device=dev))
    cfg = _roi_cfg_with(cfg, bits)
    L = load()
    fdt = _ROI_DTYPES[feat_dtype]
    if deterministic:
        wsb = L.rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(C.byref(cfg), K, fdt)
        ws = workspace(wsb, "roi")
        check(L.rsdet_roi_align_rotated_backward_deterministic(C.byref(cfg), _ROI_DTYPES[g.dtype], ptr(g), ptr(r), K, fdt,
                                                               _ptr_array(grads), ptr(ws), ws.numel(), stream_ptr()),
              "roi_align_rotated_backward (deterministic)")
        return grads
    wsb = L.rsdet_roi_align_rotated_workspace_bytes_typed(C.byref(cfg), K, 1, fdt)
    ws = workspace(wsb, "roi")
    check(L.rsdet_roi_align_rotated_backward_typed(C.byref(cfg), _ROI_DTYPES[g.dtype], ptr(g), ptr(r), K, fdt, _ptr_array(grads),
                                                   ptr(ws), ws.numel(), stream_ptr()), "roi_align_rotated_backward")
    return grads


def oriented_head_results(rois5: torch.Tensor, cls_score: torch.Tensor, bbox_pred: torch.Tensor, num_classes: int,
                          reg_class_agnostic: bool, means, stds, score_thresh: float, scale_factor=None,
                          wh_ratio_clip: float = 16 / 1000, apply_softmax: bool = True):
    """-> (dets (cap,9), labels (cap,) int64, count (1,) int32), all on device (no sync)."""
    r, s, d = _f32(rois5), _f32(cls_score), _f32(bbox_pred)
    k = r.shape[0]
    cap = max(k * num_classes, 1)
    dev = r.device
    dets = torch.empty((cap, 9), dtype=torch.float32, device=dev)
    labels = torch.empty((cap,), dtype=torch.int64, device=dev)
    cnt = torch.zeros((1,), dtype=torch.int32, device=dev)
    if k == 0:
        return dets, labels, cnt
    L = load()
    m5 = (C.c_float * 5)(*[float(v) for v in means])
    s5 = (C.c_float * 5)(*[float(v) for v in stds])
    sf = None
    if scale_factor is not None:
        sfv = [float(scale_factor)] * 4 if isinstance(scale_factor, (int, float)) else [float(v) for v in scale_factor]
        sf = (C.c_float * 4)(*sfv)
    ws = workspace(L.rsdet_oriented_head_results_workspace_bytes(k), "head")
    check(L.rsdet_oriented_head_results(ptr(r), ptr(s), ptr(d), k, int(num_classes), int(reg_class_agnostic), m5, s5,
                                        float(wh_ratio_clip), sf, float(score_thresh), int(apply_softmax), ptr(dets),
                                        ptr(labels), ptr(cnt), ptr(ws), ws.numel(), stream_ptr()), "oriented_head_results")
    return dets, labels, cnt


def voc_match(det_polys: torch.Tensor, det_img: torch.Tensor, gt_polys: torch.Tensor, gt_start: torch.Tensor,
              gt_difficult: torch.Tensor, ovthresh: float):
    """detections in descending-confidence order -> (tp uint8 (nd), fp uint8 (nd), ovmax f64 (nd), jmax int32 (nd))."""
    d = det_polys.to(torch.float64).contiguous()
    di = det_img.to(torch.int32).contiguous()
    g = gt_polys.to(torch.float64).contiguous().reshape(-1, 8)
    gs = gt_start.to(torch.int32).contiguous()
    gd = gt_difficult.to(torch.uint8).contiguous()
    nd, ng, ni = d.shape[0], g.shape[0], gs.numel() - 1
    dev = d.device
    ovmax = torch.empty((nd,), dtype=torch.float64, device=dev)
    jmax = torch.empty((nd,), dtype=torch.int32, device=dev)
    claim = torch.empty((max(ng, 1),), dtype=torch.int32, device=dev)
    tp = torch.zeros((nd,), dtype=torch.uint8, device=dev)
    fp = torch.zeros((nd,), dtype=torch.uint8, device=dev)
    check(load().rsdet_voc_match(ptr(d), ptr(di), nd, ptr(g), ptr(gs), ptr(gd), ni, ng, float(ovthresh), ptr(ovmax), ptr(jmax),
                                 ptr(claim), ptr(tp), ptr(fp), stream_ptr()), "voc_match")
    return tp, fp, ovmax, jmax


def nchw_to_nhwc(x: torch.Tensor) -> torch.Tensor:
    x = _f32(x)
    n, c, h, w = x.shape
    out = torch.empty((n, h, w, c), dtype=torch.float32, device=x.device)
    check(load().rsdet_nchw_to_nhwc(ptr(x), n, c, h, w, ptr(out), stream_ptr()), "nchw_to_nhwc")
    return out


def nhwc_to_nchw(x: torch.Tensor) -> torch.Tensor:
    x = _f32(x)
    n, h, w, c = x.shape
    out = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    check(load().rsdet_nhwc_to_nchw(ptr(x), n, c, h, w, ptr(out), stream_ptr()), "nhwc_to_nchw")
    return out


# ------------------------------------------------------------------------------- SURVEY 8(f) rank 2: RPN proposals
def rpn_proposals(cls_scores, bbox_preds, anchors, num_anchors: int, use_sigmoid: bool = True, nms_pre: int = 2000,
                  nms_post: int = 2000, nms_thresh: float = 0.8, min_bbox_size: float = 0.0,
                  means=(0., 0., 0., 0., 0., 0.), stds=(1., 1., 1., 1., 0.5, 0.5), wh_ratio_clip: float = 16 / 1000,
                  want_candidates: bool = False):
    """One image.  cls_scores[l] (A*c, H, W), bbox_preds[l] (A*6, H, W), anchors[l] (H*W*A, 4) CUDA fp32 tensors.
    -> dets (nms_post, 6) [cx,cy,w,h,theta,score] (rows past the count are zero), count (1,) int32; with
    `want_candidates` also (cand_obb, cand_hbb, cand_score, cand_level).  No host synchronisation."""
    from ._lib import RpnCfg
    cs = [_f32(t) for t in cls_scores]
    bp = [_f32(t) for t in bbox_preds]
    an = [_f32(t) for t in anchors]
    nl = len(cs)
    assert nl == len(bp) == len(an) and 1 <= nl <= 8
    cfg = RpnCfg()
    cfg.num_levels, cfg.num_anchors, cfg.use_sigmoid = nl, int(num_anchors), int(bool(use_sigmoid))
    cfg.nms_pre, cfg.nms_post, cfg.nms_thresh = int(nms_pre), int(nms_post), float(nms_thresh)
    cfg.min_bbox_size, cfg.wh_ratio_clip = float(min_bbox_size), float(wh_ratio_clip)
    for k in range(6):
        cfg.means[k], cfg.stds[k] = float(means[k]), float(stds[k])
    for l in range(nl):
        h, w = cs[l].shape[-2:]
        assert tuple(bp[l].shape[-2:]) == (h, w) and bp[l].numel() == num_anchors * 6 * h * w
        assert cs[l].numel() == num_anchors * (1 if use_sigmoid else 2) * h * w and an[l].numel() == h * w * num_anchors * 4
        cfg.height[l], cfg.width[l] = int(h), int(w)
    L = load()
    nc = L.rsdet_rpn_num_candidates(C.byref(cfg))
    if nc < 0:
        raise ValueError("rpn_proposals: bad configuration")
    dev = cs[0].device
    dets = torch.empty((int(nms_post), 6), dtype=torch.float32, device=dev)
    cnt = torch.empty((1,), dtype=torch.int32, device=dev)
    cand = (None, None, None, None)
    if want_candidates:
        cand = (torch.empty((nc, 5), dtype=torch.float32, device=dev), torch.empty((nc, 4), dtype=torch.float32, device=dev),
                torch.empty((nc,), dtype=torch.float32, device=dev), torch.empty((nc,), dtype=torch.int32, device=dev))
    vp = C.c_void_p * nl
    ws = workspace(L.rsdet_rpn_proposals_workspace_bytes(C.byref(cfg)), "rpn")
    check(L.rsdet_rpn_proposals(C.byref(cfg), vp(*[ptr(t) for t in cs]), vp(*[ptr(t) for t in bp]), vp(*[ptr(t) for t in an]),
                                ptr(dets), ptr(cnt), *[ptr(t) if t is not None else None for t in cand], ptr(ws), ws.numel(),
                                stream_ptr()), "rpn_proposals")
    return (dets, cnt) + (cand if want_candidates else ())
