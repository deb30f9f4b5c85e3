"""Jittor binding of librsdet.so -- the file a JDet maintainer drops next to `python/jdet/ops/`.

EXPERIMENTAL: Jittor is not installable in this image (no network), so these ops have never run under a live
Jittor.  What IS checked here (tests/test_jittor_adapter.py, CPU): every `cuda_header` / `cuda_src` string of this
module is extracted through a recording stand-in for `jt.code` and compiled with nvcc for sm_100a against a stub
`executor.h` and the real `include/rsdet.h` -- so the C side of every op type-checks against the C ABI it calls.

Design: every op is ONE `jt.code` whose CUDA body resolves the `extern "C"` entry point with dlopen/dlsym (no extra
link flags) and forwards Jittor's raw pointers (`in0_p`, `out0_p`, `in0_shape0`, ... -- the same glue the reference
ops use, e.g. python/jdet/ops/box_iou_rotated.py:464-485) on the legacy default stream, which is where Jittor
launches its own kernels.  The structs and prototypes come from `#include "rsdet.h"` (function pointers are
`decltype(&rsdet_...)`), never from hand-copied declarations.  Temporary memory comes from Jittor's allocator like
the reference's NMS mask (`exe.allocator->alloc/free`, python/jdet/ops/nms_rotated.py:462-464,492); the reference
synchronises the device before freeing it (:475), and so does `Scratch` here unless `SYNC_BEFORE_FREE` is switched
off after checking that Jittor's allocator recycles blocks in stream order.  A non-zero return code is raised
through Jittor's `LOGf` (a Python exception), not `abort()`.  Empty inputs and over-limit sizes are handled on the
Python side with the reference's own return values.
"""
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "librsdet.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include", "rsdet.h")
SYNC_BEFORE_FREE = True     # python/jdet/ops/nms_rotated.py:475 does cudaDeviceSynchronize before the free
MAX_NMS_BOXES = 1 << 18     # include/rsdet.h: RSDET_ELIMIT above this
MAX_MC_CANDIDATES = 1 << 20


def _header():
    return r'''
#undef out
#include <dlfcn.h>
#include <cstdint>
#include <cstring>
#include <executor.h>
#include "%s"
namespace {
inline void* rsdet_sym(const char* name) {
  static void* lib = dlopen("%s", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) LOGf << "librsdet.so:" << dlerror();
  void* f = dlsym(lib, name);
  if (!f) LOGf << "librsdet.so: missing symbol" << name;
  return f;
}
#define RSDET_FN(name) static auto fn_##name = (decltype(&name))rsdet_sym(#name)
struct Scratch {  // Jittor-owned temporary, as in nms_rotated.py:462-464
  void* p; size_t bytes, alloc;
  explicit Scratch(size_t n) : bytes(n ? n : 256) { p = exe.allocator->alloc(bytes, alloc); }
  ~Scratch() { if (%d) cudaStreamSynchronize(0); exe.allocator->free(p, bytes, alloc); }
};
inline void rsdet_check(int rc, const char* what) {
  if (rc != 0) LOGf << what << "failed: rsdet code" << rc;
}
}
''' % (INCLUDE, LIB, 1 if SYNC_BEFORE_FREE else 0)


def _jt():
    import jittor as jt  # noqa: raises ModuleNotFoundError where Jittor is absent (this image)
    return jt


def _code(shapes, dtypes, inputs, src):
    return _jt().code(shapes, dtypes, inputs, cuda_header=_header(), cuda_src=src)


# ------------------------------------------------------------------------------------------------ box transforms
def _transform(fn, x, out_cols, extra=""):
    jt = _jt()
    n = 1
    for d in x.shape[:-1]:
        n *= d
    if n == 0:
        return jt.zeros(tuple(x.shape[:-1]) + (out_cols,), dtype=x.dtype)
    y = _code((n, out_cols), x.dtype, [x], r'''
        RSDET_FN(%s);
        rsdet_check(fn_%s(in0_p, %d%s, out0_p, 0), "%s");''' % (fn, fn, n, extra, fn))
    return y.reshape(tuple(x.shape[:-1]) + (out_cols,))


def obb2poly(obboxes):
    """ops/bbox_transforms.py:612-623"""
    return _transform("rsdet_obb2poly", obboxes, 8)


def obb2hbb(obboxes):
    """ops/bbox_transforms.py:626-632"""
    return _transform("rsdet_obb2hbb", obboxes, 4)


def poly2hbb(polys):
    """ops/bbox_transforms.py:602-609"""
    return _transform("rsdet_poly2hbb", polys, 4, ", %d" % (polys.shape[-1] // 2))


def poly2obb(polys):
    """ops/bbox_transforms.py:549-575 on 4-point polygons (cv2.minAreaRect + le90): (..., 8) -> (..., 5) float64."""
    assert polys.shape[-1] == 8, "poly2obb: 4-point polygons only"
    if polys.dtype != "float64":
        polys = polys.float64()
    return _transform("rsdet_poly2obb", polys, 5)


# ------------------------------------------------------------------------------------------------ rotated IoU
def box_iou_rotated(boxes1, boxes2, version=0):
    """jdet.ops.box_iou_rotated / box_iou_rotated_v1 (box_iou_rotated.py:502-509, box_iou_rotated_v1.py:507-524)."""
    jt = _jt()
    assert boxes1.dtype == boxes2.dtype
    n1, n2 = boxes1.shape[0], boxes2.shape[0]
    if n1 == 0 or n2 == 0:
        return jt.zeros((n1, n2), dtype=boxes1.dtype)
    ious = _code((n1 * n2,), boxes1.dtype, [boxes1, boxes2], r'''
        RSDET_FN(rsdet_box_iou_rotated_workspace_bytes);
        RSDET_FN(rsdet_box_iou_rotated);
        int n1 = in0_shape0, n2 = in1_shape0;
        Scratch s(fn_rsdet_box_iou_rotated_workspace_bytes(n1, n2));
        rsdet_check(fn_rsdet_box_iou_rotated(in0_p, n1, in1_p, n2, %d, %d, out0_p, s.p, s.bytes, 0), "box_iou_rotated");'''
                 % (version, 1 if version == 1 else 0))
    return ious.reshape(n1, n2)


def box_iou_rotated_v1(boxes1, boxes2):
    return box_iou_rotated(boxes1, boxes2, 1)


def assign_wrt_overlaps(overlaps, pos_iou_thr, neg_iou_thr, min_pos_iou=0.0, match_low_quality=True, gt_max_assign_all=True,
                        gt_labels=None, assigned_labels_filled=0):
    """MaxIoUAssigner.assign_wrt_overlaps (models/boxes/assigner.py:111-170) -> (assigned_gt_inds int32, max_overlaps,
    assigned_labels int32 or None)."""
    if overlaps.numel() == 0:
        raise ValueError('No gt or proposals')
    G, n = overlaps.shape
    neg_lo, neg_hi = (neg_iou_thr if isinstance(neg_iou_thr, tuple) else (0.0, neg_iou_thr))
    ins = [overlaps] + ([gt_labels.int32()] if gt_labels is not None else [])
    outs = _code([(n,), (n,), (n,)], ["int32", overlaps.dtype, "int32"], ins, r'''
        RSDET_FN(rsdet_assign_workspace_bytes);
        RSDET_FN(rsdet_assign_wrt_overlaps);
        int G = in0_shape0, n = in0_shape1;
        Scratch s(fn_rsdet_assign_workspace_bytes(G));
        rsdet_check(fn_rsdet_assign_wrt_overlaps(in0_p, G, n, %rf, %rf, %rf, %rf, %d, %d, %s, %d, (int32_t*)out0_p, out1_p,
                                                 (int32_t*)out2_p, s.p, s.bytes, 0), "assign_wrt_overlaps");'''
                 % (float(pos_iou_thr), float(neg_lo), float(neg_hi), float(min_pos_iou), int(match_low_quality),
                    int(gt_max_assign_all), "(const int32_t*)in1_p" if gt_labels is not None else "nullptr",
                    int(assigned_labels_filled)))
    return outs[0], outs[1], (outs[2] if gt_labels is not None else None)


# ------------------------------------------------------------------------------------------------ horizontal IoU
def bbox_overlaps(bboxes1, bboxes2):
    """BboxOverlaps2D (mode='iou', not aligned; models/boxes/iou_calculator.py): (n1,4) x (n2,4) -> (n1,n2)."""
    jt = _jt()
    n1, n2 = bboxes1.shape[0], bboxes2.shape[0]
    if n1 == 0 or n2 == 0:
        return jt.zeros((n1, n2), dtype="float32")
    ious = _code((n1 * n2,), "float32", [bboxes1, bboxes2], r'''
        RSDET_FN(rsdet_bbox_overlaps);
        rsdet_check(fn_rsdet_bbox_overlaps(in0_p, in0_shape0, in1_p, in1_shape0, out0_p, 0), "bbox_overlaps");''')
    return ious.reshape(n1, n2)


def assign_hbb(gt_hbb, anchors, pos_iou_thr, neg_iou_thr, min_pos_iou=0.0, match_low_quality=True, gt_max_assign_all=True,
               gt_labels=None, assigned_labels_filled=0, valid=None):
    """assign_wrt_overlaps(bbox_overlaps(gt_hbb, anchors), ...) fused (rsdet_assign_hbb); `valid` is an optional uint8
    (n,) mask (anchor_inside_flags).  -> (assigned_gt_inds int32, max_overlaps, assigned_labels int32 or None)."""
    G, n = gt_hbb.shape[0], anchors.shape[0]
    if G == 0 or n == 0:
        raise ValueError('No gt or proposals')
    neg_lo, neg_hi = (neg_iou_thr if isinstance(neg_iou_thr, tuple) else (0.0, neg_iou_thr))
    ins = [gt_hbb, anchors]
    labels_in = valid_in = "nullptr"
    if gt_labels is not None:
        labels_in = "(const int32_t*)in%d_p" % len(ins)
        ins.append(gt_labels.int32())
    if valid is not None:
        valid_in = "(const uint8_t*)in%d_p" % len(ins)
        ins.append(valid)
    outs = _code([(n,), (n,), (n,)], ["int32", "float32", "int32"], ins, r'''
        RSDET_FN(rsdet_assign_hbb_workspace_bytes);
        RSDET_FN(rsdet_assign_hbb);
        int G = in0_shape0, n = in1_shape0;
        Scratch s(fn_rsdet_assign_hbb_workspace_bytes(G, n));
        rsdet_check(fn_rsdet_assign_hbb(in0_p, G, in1_p, n, %s, %rf, %rf, %rf, %rf, %d, %d, %s, %d, (int32_t*)out0_p, out1_p,
                                        (int32_t*)out2_p, s.p, s.bytes, 0), "assign_hbb");'''
                 % (valid_in, float(pos_iou_thr), float(neg_lo), float(neg_hi), float(min_pos_iou), int(match_low_quality),
                    int(gt_max_assign_all), labels_in, int(assigned_labels_filled)))
    return outs[0], outs[1], (outs[2] if gt_labels is not None else None)


# ------------------------------------------------------------------------------------------------ NMS family
def _nms_keep(kind, dets, scores, labels, thr):
    """bool keep mask in ORIGINAL index space (nms_rotated_cuda's `keep`, nms_rotated.py:506-513)."""
    n = dets.shape[0]
    if n > MAX_NMS_BOXES:
        raise ValueError("rsdet NMS: at most %d boxes per call (got %d)" % (MAX_NMS_BOXES, n))
    ins = [dets, scores] + ([labels.int32()] if labels is not None else [])
    return _code((n,), "uint8", ins, r'''
        RSDET_FN(rsdet_nms_workspace_bytes);
        RSDET_FN(rsdet_nms);
        int n = in0_shape0;
        Scratch s(fn_rsdet_nms_workspace_bytes(%d, n));
        rsdet_check(fn_rsdet_nms(%d, in0_p, in1_p, %s, n, %r, nullptr, 0, (uint8_t*)out0_p, nullptr, nullptr, nullptr,
                                 s.p, s.bytes, 0), "nms");'''
                 % (kind, kind, "(const int32_t*)in2_p" if labels is not None else "nullptr", float(thr))).bool()


def nms_rotated(dets, scores, iou_threshold):
    """nms_rotated.py:527-538"""
    jt = _jt()
    if dets.numel() == 0:
        return jt.array([])
    assert dets.numel() > 0 and dets.ndim == 2 and dets.dtype == scores.dtype
    return jt.where(_nms_keep(0, dets, scores, None, iou_threshold))[0]


def ml_nms_rotated(dets, scores, labels, iou_threshold):
    """nms_rotated.py:515-525"""
    jt = _jt()
    assert dets.numel() > 0 and dets.ndim == 2 and dets.dtype == scores.dtype
    return jt.where(_nms_keep(0, dets, scores, labels, iou_threshold))[0]


def _nms_sorted_keep(kind, dets_sorted, thr):
    """keep mask over rows that are ALREADY in descending-score order (the contract of nms_rotated_cpu/cuda,
    nms_rotated.py:495-513: `dets[order_t]` in, bool keep out): positions serve as scores."""
    jt = _jt()
    n = dets_sorted.shape[0]
    scores = (n - jt.arange(n)).float32()
    box_len = dets_sorted.shape[1]
    labels = dets_sorted[:, 5] if box_len == 6 else None
    return _nms_keep(kind, dets_sorted[:, :5], scores, labels, thr)


def nms_rotated_cuda(dets_sorted, order_t, iou_threshold, box_length=5):
    """nms_rotated.py:506-513 (suppression rule IoU > thr)"""
    return _nms_sorted_keep(0, dets_sorted, iou_threshold)


def nms_rotated_cpu(dets_sorted, order_t, iou_threshold, box_length=5):
    """nms_rotated.py:495-504 (suppression rule IoU >= thr); runs on the device like everything here"""
    return _nms_sorted_keep(1, dets_sorted, iou_threshold)


def poly_nms(boxes, nms_overlap_thresh):
    """nms_poly.py:187-232 -> order_t[keep]"""
    assert boxes.ndim == 2 and boxes.shape[1] == 9
    scores = boxes[:, 8]
    order_t, _ = scores.argsort(0, descending=True)
    keep = _nms_keep(2, boxes[:, :8], scores, None, nms_overlap_thresh)
    return order_t[keep[order_t]]


def multiclass_poly_nms(bboxes, scores, labels, thresh):
    """nms_poly.py:234-245: class separation by the coordinate offset trick == label-gated NMS"""
    jt = _jt()
    if bboxes.shape[0] == 0:
        return jt.zeros((0, 9), dtype=bboxes.dtype), labels
    order_t, _ = scores.argsort(0, descending=True)
    keep_mask = _nms_keep(2, bboxes, scores, labels, thresh)
    keep = order_t[keep_mask[order_t]]
    return jt.concat([bboxes[keep], scores[keep][:, None]], dim=1), labels[keep]


def multiclass_nms_rotated(multi_bboxes, multi_scores, score_thr, nms_cfg, max_num=-1, score_factors=None):
    """jdet.ops.nms_rotated.multiclass_nms_rotated (nms_rotated.py:540-596) as ONE jt.code: candidate selection,
    per-class NMS through the shared decision matrix, score sort and top-k on the device.  Returns
    (dets (k,6), labels (k,)) like the reference; k is read back once (the reference syncs in jt.where)."""
    jt = _jt()
    n, C = multi_scores.shape[0], multi_scores.shape[1] - 1
    if n == 0:
        return jt.zeros((0, 6)), jt.zeros((0,)).int32()
    cap = n * C  # the C entry point needs n*C rows of output whatever max_num is
    if cap > MAX_MC_CANDIDATES or n > MAX_NMS_BOXES:
        raise ValueError("rsdet multiclass NMS: n * classes <= %d (got %d x %d)" % (MAX_MC_CANDIDATES, n, C))
    ins = [multi_bboxes, multi_scores] + ([score_factors] if score_factors is not None else [])
    dets, labels, cnt = _code([(cap, 6), (cap,), (1,)], [multi_bboxes.dtype, "int32", "int32"], ins, r'''
        RSDET_FN(rsdet_multiclass_nms_rotated_workspace_bytes);
        RSDET_FN(rsdet_multiclass_nms_rotated);
        int n = in1_shape0, C = in1_shape1 - 1;
        Scratch s(fn_rsdet_multiclass_nms_rotated_workspace_bytes(n, C));
        rsdet_check(fn_rsdet_multiclass_nms_rotated(in0_p, in0_shape1, in1_p, n, C, %rf, %rf, %d, %s, out0_p, (int32_t*)out1_p,
                                                    (int32_t*)out2_p, s.p, s.bytes, 0), "multiclass_nms_rotated");'''
                            % (float(score_thr), float(nms_cfg.get('iou_thr', 0.1)), int(max_num),
                               "in2_p" if score_factors is not None else "nullptr"))
    k = int(cnt.item())
    return dets[:k], labels[:k]


# ------------------------------------------------------------------------------------------------ RoIAlignRotated
def _roi_cfg_src(num_levels, scales, ph, pw, sampling_ratio, version, extend_h, extend_w, finest_scale):
    """fills an `rsdet_roi_align_cfg cfg` (the struct of include/rsdet.h) from the feature inputs in0..in{L-1}"""
    src = ["        rsdet_roi_align_cfg cfg; memset(&cfg, 0, sizeof cfg);",
           "        cfg.num_levels = %d; cfg.batch = in0_shape0; cfg.channels = in0_shape1;" % num_levels]
    for l in range(num_levels):
        src.append("        cfg.height[%d] = in%d_shape2; cfg.width[%d] = in%d_shape3; cfg.spatial_scale[%d] = %rf;"
                   % (l, l, l, l, l, float(scales[l])))
    src.append("        cfg.pooled_h = %d; cfg.pooled_w = %d; cfg.sampling_ratio = %d; cfg.version = %d;"
               % (ph, pw, sampling_ratio, version))
    src.append("        cfg.extend_w = %rf; cfg.extend_h = %rf; cfg.finest_scale = %rf;"
               % (float(extend_w), float(extend_h), float(finest_scale)))
    src.append("        RSDET_FN(rsdet_roi_align_rotated_workspace_bytes);")
    return "\n".join(src) + "\n"


def _is_half(var):
    return str(var.dtype) == "float16"


def _roi_half_fwd_src(L, what):
    """forward body for float16 maps in0..in{L-1} and fp32 rois in{L}: the typed entry point, float16 output"""
    return r'''
        RSDET_FN(rsdet_roi_align_rotated_workspace_bytes_typed);
        RSDET_FN(rsdet_roi_align_rotated_forward_typed);
        int K = in%d_shape0;
        Scratch s(fn_rsdet_roi_align_rotated_workspace_bytes_typed(&cfg, K, 0, RSDET_DTYPE_F16));
        const void* feats[RSDET_MAX_LEVELS] = {%s};
        rsdet_check(fn_rsdet_roi_align_rotated_forward_typed(&cfg, RSDET_DTYPE_F16, feats, (const float*)in%d_p, K, RSDET_DTYPE_F16,
                                                             out0_p, nullptr, s.p, s.bytes, 0), "%s");''' % (
        L, ", ".join("in%d_p" % l for l in range(L)), L, what)


def _roi_half_bwd_src(L, grad_half, what):
    """backward body: float16 gradient maps out0..out{L-1} from grad_out in{L+1} (float16 or fp32) and rois in{L}"""
    return r'''
        RSDET_FN(rsdet_roi_align_rotated_workspace_bytes_typed);
        RSDET_FN(rsdet_roi_align_rotated_backward_typed);
        int K = in%d_shape0;
        Scratch s(fn_rsdet_roi_align_rotated_workspace_bytes_typed(&cfg, K, 1, RSDET_DTYPE_F16));
        void* grads[RSDET_MAX_LEVELS] = {%s};
        rsdet_check(fn_rsdet_roi_align_rotated_backward_typed(&cfg, %s, in%d_p, (const float*)in%d_p, K, RSDET_DTYPE_F16, grads,
                                                              s.p, s.bytes, 0), "%s");''' % (
        L, ", ".join("out%d_p" % l for l in range(L)), "RSDET_DTYPE_F16" if grad_half else "RSDET_DTYPE_F32", L + 1, L, what)


def make_roi_align(version):
    """Returns the jt.Function class replacing _RotatedROIAlign(_v1) (roi_align_rotated_v1.py:300-353):
    `.apply(input, rois, output_size, spatial_scale, sampling_ratio)`; grad -> (input_grad, None)."""
    jt = _jt()

    class _Fn(jt.Function):
        def execute(self, input, rois, output_size, spatial_scale, sampling_ratio):
            self.input, self.rois = input, rois
            assert rois.shape[1] == 6
            self.cfg = _roi_cfg_src(1, [spatial_scale], int(output_size[0]), int(output_size[1]), int(sampling_ratio), version,
                                    1.0, 1.0, 56.0)
            shape = (rois.shape[0], input.shape[1], output_size[0], output_size[1])
            if rois.shape[0] == 0:
                return jt.zeros(shape, dtype=input.dtype)
            if _is_half(input):      # float16 maps are read natively (include/rsdet.h); rois stay fp32
                if str(rois.dtype) != "float32":
                    self.rois = rois = rois.float32()
                return _code(shape, input.dtype, [input, rois], self.cfg + _roi_half_fwd_src(1, "roi_align_rotated_forward"))
            return _code(shape, input.dtype, [input, rois], self.cfg + r'''
        RSDET_FN(rsdet_roi_align_rotated_forward);
        int K = in1_shape0;
        Scratch s(fn_rsdet_roi_align_rotated_workspace_bytes(&cfg, K, 0));
        const float* feats[RSDET_MAX_LEVELS] = {in0_p};
        rsdet_check(fn_rsdet_roi_align_rotated_forward(&cfg, feats, in1_p, K, out0_p, nullptr, s.p, s.bytes, 0),
                    "roi_align_rotated_forward");''')

        def grad(self, output_grad):
            input, rois = self.input, self.rois
            if _is_half(input):
                g = _code(input.shape, input.dtype, [input, rois, output_grad],
                          self.cfg + _roi_half_bwd_src(1, _is_half(output_grad), "roi_align_rotated_backward"))
                return g, None
            g = _code(input.shape, input.dtype, [input, rois, output_grad], self.cfg + r'''
        RSDET_FN(rsdet_roi_align_rotated_backward);
        int K = in1_shape0;
        Scratch s(fn_rsdet_roi_align_rotated_workspace_bytes(&cfg, K, 1));
        float* grads[RSDET_MAX_LEVELS] = {out0_p};
        rsdet_check(fn_rsdet_roi_align_rotated_backward(&cfg, in2_p, in1_p, K, grads, s.p, s.bytes, 0),
                    "roi_align_rotated_backward");''')
            return g, None

    return _Fn


def make_fused_extractor(version=1):
    """The whole `OrientedSingleRoIExtractor.execute` level loop (models/roi_extractors/oriented_single_level.py:91-114:
    roi_rescale, map_roi_levels, per-level gather -> op -> masked scatter-add) as ONE launch over all levels:
    `.apply(feat_0, ..., feat_{L-1}, rois, featmap_strides, output_size, sampling_ratio, extend_factor, finest_scale)`.
    grad -> one gradient per feature level followed by None for rois and the constants."""
    jt = _jt()

    class _Fused(jt.Function):
        def execute(self, *args):
            *head, strides, output_size, sampling_ratio, extend_factor, finest_scale = args
            feats, rois = list(head[:-1]), head[-1]
            L = len(feats)
            assert 1 <= L <= 8 and rois.shape[1] == 6
            self.feats, self.rois, self.nconst = feats, rois, 5
            ph, pw = (output_size, output_size) if isinstance(output_size, int) else output_size
            eh, ew = (1.0, 1.0) if L == 1 else extend_factor           # len(feats) == 1: no extension (:92-93)
            self.cfg = _roi_cfg_src(L, [1.0 / s for s in strides[:L]], int(ph), int(pw), int(sampling_ratio), version, eh, ew,
                                    finest_scale)
            shape = (rois.shape[0], feats[0].shape[1], ph, pw)
            if rois.shape[0] == 0:
                return jt.zeros(shape, dtype=feats[0].dtype)
            if any(_is_half(f) for f in feats):
                if not all(_is_half(f) for f in feats):
                    raise ValueError("rsdet RoIAlignRotated: feature levels mix float16 with another dtype")
                if str(rois.dtype) != "float32":
                    self.rois = rois = rois.float32()
                return _code(shape, feats[0].dtype, feats + [rois],
                             self.cfg + _roi_half_fwd_src(L, "roi_align_rotated_forward (fused levels)"))
            ptrs = ", ".join("in%d_p" % l for l in range(L))
            return _code(shape, feats[0].dtype, feats + [rois], self.cfg + r'''
        RSDET_FN(rsdet_roi_align_rotated_forward);
        int K = in%d_shape0;
        Scratch s(fn_rsdet_roi_align_rotated_workspace_bytes(&cfg, K, 0));
        const float* feats[RSDET_MAX_LEVELS] = {%s};
        rsdet_check(fn_rsdet_roi_align_rotated_forward(&cfg, feats, in%d_p, K, out0_p, nullptr, s.p, s.bytes, 0),
                    "roi_align_rotated_forward (fused levels)");''' % (L, ptrs, L))

        def grad(self, output_grad):
            feats, rois = self.feats, self.rois
            L = len(feats)
            if _is_half(feats[0]):
                gs = _code([f.shape for f in feats], [f.dtype for f in feats], feats + [rois, output_grad],
                           self.cfg + _roi_half_bwd_src(L, _is_half(output_grad), "roi_align_rotated_backward (fused levels)"))
                gs = list(gs) if isinstance(gs, (list, tuple)) else [gs]
                return tuple(gs) + (None,) * (1 + self.nconst)
            outs = ", ".join("out%d_p" % l for l in range(L))
            gs = _code([f.shape for f in feats], [f.dtype for f in feats], feats + [rois, output_grad], self.cfg + r'''
        RSDET_FN(rsdet_roi_align_rotated_backward);
        int K = in%d_shape0;
        Scratch s(fn_rsdet_roi_align_rotated_workspace_bytes(&cfg, K, 1));
        float* grads[RSDET_MAX_LEVELS] = {%s};
        rsdet_check(fn_rsdet_roi_align_rotated_backward(&cfg, in%d_p, in%d_p, K, grads, s.p, s.bytes, 0),
                    "roi_align_rotated_backward (fused levels)");''' % (L, outs, L + 1, L))
            gs = list(gs) if isinstance(gs, (list, tuple)) else [gs]
            return tuple(gs) + (None,) * (1 + self.nconst)

    return _Fused


# ------------------------------------------------------------------------------------------------ oriented RPN proposals
def rpn_proposals(cls_scores, bbox_preds, mlvl_anchors, num_anchors, use_sigmoid=True, nms_pre=2000, nms_post=2000,
                  nms_thresh=0.8, min_bbox_size=0, means=(0.,) * 6, stds=(1., 1., 1., 1., 0.5, 0.5), wh_ratio_clip=16 / 1000):
    """OrientedRPNHead._get_bboxes_single (oriented_rpn_head.py:136-216) as one jt.code over 3L inputs."""
    L = len(cls_scores)
    assert 1 <= L <= 8
    ins = list(cls_scores) + list(bbox_preds) + list(mlvl_anchors)
    lv = "".join("        cfg.height[%d] = in%d_shape1; cfg.width[%d] = in%d_shape2; cls[%d] = in%d_p; reg[%d] = in%d_p; anc[%d] = in%d_p;\n"
                 % (l, l, l, l, l, l, l, L + l, l, 2 * L + l) for l in range(L))
    dets, cnt = _code([(nms_post, 6), (1,)], [cls_scores[0].dtype, "int32"], ins, r'''
        rsdet_rpn_cfg cfg; memset(&cfg, 0, sizeof cfg);
        const float *cls[8], *reg[8], *anc[8];
        cfg.num_levels = %d; cfg.num_anchors = %d; cfg.use_sigmoid = %d; cfg.nms_pre = %d; cfg.nms_post = %d;
        cfg.nms_thresh = %r; cfg.min_bbox_size = %rf; cfg.wh_ratio_clip = %rf;
        const float mm[6] = {%s}, ss[6] = {%s};
        for (int k = 0; k < 6; k++) { cfg.means[k] = mm[k]; cfg.stds[k] = ss[k]; }
%s
        RSDET_FN(rsdet_rpn_proposals_workspace_bytes);
        RSDET_FN(rsdet_rpn_proposals);
        Scratch s(fn_rsdet_rpn_proposals_workspace_bytes(&cfg));
        rsdet_check(fn_rsdet_rpn_proposals(&cfg, cls, reg, anc, out0_p, (int32_t*)out1_p, nullptr, nullptr, nullptr, nullptr,
                                           s.p, s.bytes, 0), "rpn_proposals");'''
                      % (L, num_anchors, int(use_sigmoid), nms_pre, nms_post, float(nms_thresh), float(min_bbox_size),
                         float(wh_ratio_clip), ", ".join("%rf" % float(m) for m in means),
                         ", ".join("%rf" % float(v) for v in stds), lv))
    return dets[:int(cnt.item())]
