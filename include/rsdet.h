/*
 * rsdet.h -- C ABI of librsdet.so: the B200 (sm_100a) rotated-box hot path for JDet / RS_detection.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI: every op is a
 * C++/CUDA string handed to Jittor's `jt.code`, which passes raw `in<i>_p / out0_p` pointers and
 * shapes.  Each entry point below replaces one such JIT body (cited `file:line`, relative to the
 * reference's `python/jdet/`), and is what a `jt.code` one-liner / ctypes stub binds (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`; the caller owns all memory
 *     (inputs, outputs, workspace); the library never allocates, frees or retains pointers;
 *   - all work is enqueued on `stream` (a `cudaStream_t`, passed as void*; NULL = legacy default
 *     stream, which is what Jittor uses); no entry point synchronises the host;
 *   - return value: 0 = RSDET_OK, negative = RSDET_E* argument error, positive = cudaError_t;
 *   - workspace: `*_workspace_bytes()` returns the exact requirement for the given sizes; pass at
 *     least that many bytes, 256-byte aligned;
 *   - box formats: obb = [cx, cy, w, h, theta(rad)], roi = [batch, cx, cy, w, h, theta],
 *     poly = [x1,y1,...,x4,y4]; fp32 unless stated; row-major, densely packed.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns a CUDA error.
 */
#ifndef RSDET_H_
#define RSDET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSDET_OK 0
#define RSDET_EINVAL (-1)     /* bad size / flag / null pointer */
#define RSDET_EWORKSPACE (-2) /* workspace too small */
#define RSDET_ELIMIT (-3)     /* size above a documented limit */

#define RSDET_MAX_LEVELS 8

/* library version (major*10000 + minor*100 + patch) and error text */
int rsdet_version(void);
const char* rsdet_error_string(int code);

/* ---------------------------------------------------------------- box transforms
 * ops/bbox_transforms.py:612-623 (obb2poly), :626-632 (obb2hbb), :602-609 (poly2hbb).  n rows. */
int rsdet_obb2poly(const float* obb, int n, float* poly, void* stream);
int rsdet_obb2hbb(const float* obb, int n, float* hbb, void* stream);
int rsdet_poly2hbb(const float* poly, int n, int num_points, float* hbb, void* stream);

/* ---------------------------------------------------------------- rotated IoU
 * ops/box_iou_rotated.py:502-509 + kernel :413-461 (version 0);
 * ops/box_iou_rotated_v1.py:507-524 + kernel :418-466 (version 1: clockwise-positive angle).
 * boxes1 (n1,5), boxes2 (n2,5) -> ious (n1,n2).  `zero_tiny` != 0 applies the v1 wrapper's
 * guard (rows/cols whose min(w,h) < 1e-3 are zeroed, box_iou_rotated_v1.py:515-522). */
size_t rsdet_box_iou_rotated_workspace_bytes(int n1, int n2);
int rsdet_box_iou_rotated(const float* boxes1, int n1, const float* boxes2, int n2, int version, int zero_tiny,
                          float* ious, void* workspace, size_t workspace_bytes, void* stream);

/* models/boxes/assigner.py:111-170 (MaxIoUAssigner.assign_wrt_overlaps) on a (num_gts, n) overlaps
 * matrix: per-column max/argmax (first maximum wins), neg/pos thresholds, optional low-quality
 * matching (`match_low_quality`, `gt_max_assign_all`).  neg_lo/neg_hi: negatives are
 * neg_lo <= max < neg_hi (a scalar neg_iou_thr t is passed as (0, t)).  gt_labels may be NULL
 * (then assigned_labels may be NULL).  Outputs: assigned_gt_inds int32 (n), max_overlaps fp32 (n),
 * assigned_labels int32 (n). */
size_t rsdet_assign_workspace_bytes(int num_gts);
int rsdet_assign_wrt_overlaps(const float* overlaps, int num_gts, int n, float pos_iou_thr, float neg_lo, float neg_hi,
                              float min_pos_iou, int match_low_quality, int gt_max_assign_all, const int32_t* gt_labels,
                              int32_t labels_fill, int32_t* assigned_gt_inds, float* max_overlaps,
                              int32_t* assigned_labels, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- NMS (rotated / poly / merge)
 * One engine, one pair predicate per `kind`: */
#define RSDET_NMS_ROTATED 0 /* dets (n,5) fp32 obb; suppress IoU >  thr: ops/nms_rotated.py:353-411,450-493 */
#define RSDET_NMS_ROTATED_GE 1 /* same, suppress IoU >= thr (the CPU body, ops/nms_rotated.py:414-449)        */
#define RSDET_NMS_POLY 2    /* dets (n,8) fp32 quads, devPolyIoU > thr: ops/nms_poly.py:113-185,187-232       */
#define RSDET_NMS_MERGE 3   /* dets (n,8) fp64 quads in scene coords; hbb prefilter then polygon IoU > thr:
                               data/devkits/result_merge.py:66-127 + ops/nms_poly.py:247-252              */
#define RSDET_NMS_HBB 4     /* dets (n,4) fp64 [x1,y1,x2,y2]; suppress IoU >= thr (merge.py:14-27)         */
#define RSDET_NMS_HBB_P1_F64 6 /* dets (n,4) fp64, "+1" widths, survivors IoU <= thr: py_cpu_nms,
                               data/devkits/result_merge.py:143-174 (mergebyrec)                          */
#define RSDET_NMS_HBB_P1 5  /* dets (n,4) fp32 [x1,y1,x2,y2], "+1" widths; suppress IoU > thr: jt.nms as called
                               by models/roi_heads/oriented_rpn_head.py:208 (Jittor 1.3.4.7 misc.py)      */

/* Greedy NMS in descending-score order, independently inside each label group (labels == NULL: one
 * group).  Equivalent to the reference's label-gated IoU (ops/nms_rotated.py:281-286) and to one
 * reference call per class / per scene file.
 *   dets    : (n, row_floats(kind)) of fp32 or fp64 as the kind says
 *   scores  : (n) fp32, or fp64 for MERGE/HBB/HBB_P1_F64
 *   labels  : (n) int32 group ids (any values) or NULL
 *   thr     : scalar threshold, used when thr_per_label == NULL
 *   thr_per_label : optional device array indexed by label value (0 <= label < num_thr)
 *                   (result_merge.py:26-27 per-class thresholds)
 * Outputs (any may be NULL):
 *   keep_mask     uint8 (n), 1 = kept, ORIGINAL index space  (the `keep` bool Var of nms_rotated_cuda)
 *   keep_sorted_idx int64 (n): kept ORIGINAL indices in ascending index order  (jt.where(keep)[0])
 *   keep_score_idx  int64 (n): kept ORIGINAL indices in descending score order (order_t[keep], poly_nms;
 *                              py_cpu_nms_poly_fast's python list)
 *   num_keep      int32 (1) device counter
 * Score ties are broken by lower original index first (the reference leaves this unspecified).
 * Limit: n <= 2^18 boxes per call (RSDET_ELIMIT above; the workspace query then returns 0). */
size_t rsdet_nms_workspace_bytes(int kind, int n);
int rsdet_nms(int kind, const void* dets, const void* scores, const int32_t* labels, int n, double thr,
              const double* thr_per_label, int num_thr, uint8_t* keep_mask, int64_t* keep_sorted_idx,
              int64_t* keep_score_idx, int32_t* num_keep, void* workspace, size_t workspace_bytes, void* stream);

/* ops/nms_rotated.py:540-596 (multiclass_nms_rotated) fused: candidate selection scores[:,1:] >
 * score_thr (column 0 = background), label-aware rotated NMS (IoU > iou_thr), descending-score
 * ordering and top-`max_num` truncation (max_num < 0 reproduces the reference's `keep.size(0) >
 * max_num` slice `inds[:max_num]`, i.e. drops the last detection).
 *   multi_bboxes : (n,5) or (n,5*(num_classes+1)) as bbox_dim says;  multi_scores : (n,num_classes+1)
 *   score_factors: (n) or NULL
 *   out_dets (cap,6) [cx,cy,w,h,theta,score], out_labels int32 (cap), out_count int32 (1);
 *   cap = n*num_classes rows must be available; n*num_classes <= 2^20 (RSDET_ELIMIT above). */
size_t rsdet_multiclass_nms_rotated_workspace_bytes(int n, int num_classes);
int rsdet_multiclass_nms_rotated(const float* multi_bboxes, int bbox_dim, const float* multi_scores, int n,
                                 int num_classes, float score_thr, float iou_thr, int max_num,
                                 const float* score_factors, float* out_dets, int32_t* out_labels, int32_t* out_count,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- RoIAlignRotated
 * ops/roi_align_rotated_v1.py:300-351 (kernels :71-147, :193-298) and ops/roi_align_rotated.py:256-307,
 * plus the level mapping / RoI extension / per-level scatter of
 * models/roi_extractors/oriented_single_level.py:53-114 fused into ONE launch. */
typedef struct {
    int num_levels;                        /* 1..RSDET_MAX_LEVELS; 1 = plain single-map op            */
    int batch;                             /* N of every feature map                                  */
    int channels;                          /* C (multiple of 4)                                       */
    int height[RSDET_MAX_LEVELS];
    int width[RSDET_MAX_LEVELS];
    float spatial_scale[RSDET_MAX_LEVELS]; /* 1/stride                                                */
    int pooled_h, pooled_w;                /* output_size                                             */
    int sampling_ratio;                    /* >0 fixed grid, <=0 adaptive ceil(roi/pooled)            */
    int version;                           /* 1 = ROIAlignRotated_v1 (-0.5, clockwise), 0 = v0        */
    float extend_w, extend_h;              /* RoI extension (1.2, 1.4 in orcnn configs); 1,1 = none   */
    float finest_scale;                    /* 56; used when num_levels > 1                            */
    int channels_last;                     /* features (and grads) are NHWC instead of NCHW           */
} rsdet_roi_align_cfg;

/* feats[l]: (N,C,H_l,W_l) fp32 (NCHW, or NHWC when channels_last); rois (K,6);
 * out (K,C,ph,pw) fp32 -- always the reference's NCHW-style layout.  levels_out: optional int32 (K).
 *
 * Alignment.  fp32 / int32 pointers need only their natural 4-byte alignment; 16-byte alignment selects faster
 * kernels, never different results beyond what is stated here.  The fast path is C % 4 == 0, sampling_ratio > 0 and
 * pooled_h * pooled_w * sampling_ratio^2 <= 1024; outside it every call runs the scalar generic kernel.
 *   forward  feats[l]    NCHW: read by the NCHW->NHWC copy, which uses 16-byte loads where the map allows them.
 *                        NHWC: the fast kernels read 16-byte vectors from each map's base; if any base is not 16-byte
 *                        aligned the call runs the generic kernel (same results to the forward tolerance, slower).
 *            rois        read as scalars.
 *            out         16-byte aligned: the 7x7 / sampling_ratio 2 / C % 256 == 0 geometry runs the persistent kernel
 *                        and the kernels write with bulk (TMA) stores; otherwise a one-CTA-per-RoI kernel with scalar
 *                        stores.  Bit-identical results either way.
 *            levels_out  written as scalars.
 *   backward grad_out    16-byte aligned: staged with 16-byte loads; otherwise with scalar loads.  Same results.
 *            grad_feats  NCHW: written by the NHWC->NCHW copy, which uses 16-byte stores where the map allows them.
 *                        NHWC: the fast kernel accumulates with 16-byte vector reductions from each map's base; if
 *                        any base is not 16-byte aligned the call runs the generic kernel (scalar atomics).
 * Backward results are sums of atomics in an unspecified order: equal across these paths to the backward tolerance.
 * rsdet_roi_align_rotated_backward_deterministic (below) sums in the reference's order instead: the same bits every run. */
size_t rsdet_roi_align_rotated_workspace_bytes(const rsdet_roi_align_cfg* cfg, int num_rois, int backward);
int rsdet_roi_align_rotated_forward(const rsdet_roi_align_cfg* cfg, const float* const* feats_host, const float* rois,
                                    int num_rois, float* out, int32_t* levels_out, void* workspace,
                                    size_t workspace_bytes, void* stream);
/* grad_out (K,C,ph,pw) -> grad_feats[l] (N,C,H_l,W_l), fully overwritten (zero-filled + accumulated). */
int rsdet_roi_align_rotated_backward(const rsdet_roi_align_cfg* cfg, const float* grad_out, const float* rois,
                                     int num_rois, float* const* grad_feats_host, void* workspace,
                                     size_t workspace_bytes, void* stream);

/* Half-precision feature pyramids.  The three calls above are these with RSDET_DTYPE_F32 everywhere.
 *   feat_dtype      element type of every feats[l] (forward) and grad_feats[l] (backward): F32, F16 or BF16.
 *   out_dtype       forward output: F32 or feat_dtype.
 *   grad_out_dtype  backward grad_out: F32 or feat_dtype.
 * rois stay fp32 and levels_out int32.  Any other dtype, or an out_dtype / grad_out_dtype that is neither F32 nor
 * feat_dtype, returns RSDET_EINVAL before anything is launched (the workspace query returns 0).
 * Arithmetic.  Every fp16 / bf16 value converts exactly to fp32; after that the computation is the fp32 one unchanged
 * (same sample positions, tap lists, tap order and FMA order, fp32 accumulation).  Hence a forward with fp32 output is
 * bit-identical to the fp32 call on the maps converted to fp32, in the same layout and with buffers of the same
 * alignment class, and a forward with half output is that result rounded once to nearest-even.  The backward
 * accumulates in fp32 workspace maps and writes the gradient maps once, rounded to nearest-even; its atomic order is
 * unspecified as above.  The workspace query counts those accumulators (forward: a half NHWC copy of NCHW maps, half
 * the bytes of the fp32 copy).
 * Alignment with 2-byte maps.  The fast kernels read four channels (8 bytes) at a time: channels-last feature maps
 * (forward) need 8-byte aligned bases, otherwise the call runs the generic kernel.  Half gradient maps are written by a
 * transpose (NCHW) or a conversion pass (NHWC) from the fp32 accumulators, so no alignment selects a different kernel
 * for them.  out and grad_out follow the rules above: a 16-byte aligned out takes the persistent kernel and bulk stores;
 * a grad_out whose base is aligned to four elements (8 bytes when half) is staged with vector loads.  Results do not
 * depend on alignment beyond what is stated above for fp32. */
#define RSDET_DTYPE_F32 0
#define RSDET_DTYPE_F16 1
#define RSDET_DTYPE_BF16 2
size_t rsdet_roi_align_rotated_workspace_bytes_typed(const rsdet_roi_align_cfg* cfg, int num_rois, int backward,
                                                     int feat_dtype);
int rsdet_roi_align_rotated_forward_typed(const rsdet_roi_align_cfg* cfg, int feat_dtype, const void* const* feats_host,
                                          const float* rois, int num_rois, int out_dtype, void* out, int32_t* levels_out,
                                          void* workspace, size_t workspace_bytes, void* stream);
int rsdet_roi_align_rotated_backward_typed(const rsdet_roi_align_cfg* cfg, int grad_out_dtype, const void* grad_out,
                                           const float* rois, int num_rois, int feat_dtype, void* const* grad_feats_host,
                                           void* workspace, size_t workspace_bytes, void* stream);

/* Deterministic backward: same arguments, dtypes and output as rsdet_roi_align_rotated_backward_typed; the caller picks it.
 *   Summation order.  Every gradient-map element (level, image, channel, pixel) is the fp32 sum, starting from +0, of
 *     (top * w) / count, one term per (RoI, bin, sample, tap) whose sample is in range, taken in the reference's order
 *     (roi_align_rotated_v1.py:193-298): RoI index, bin row, bin column, sample row, sample column, tap lt, rt, lb, rb.
 *     Every multiply, divide and add is rounded separately, and taps that land on the same pixel are not merged.  Terms
 *     of weight 0 are dropped (adding +-0 to such a sum changes no bit), as are RoIs whose batch index is outside
 *     [0, batch).  Half maps get that fp32 value rounded once to nearest-even; a half grad_out converts exactly first.
 *   Consequences.  The same bits on every run, stream, CUDA-graph replay, layout (NCHW / channels-last), buffer alignment
 *     and batch split (a batched call equals per-image calls with each image's RoIs in the same relative order); and,
 *     for finite grad_out, bit-identity with the reference's arithmetic wherever the device's cosf / sinf agree with the
 *     host's (always at theta = 0).
 *   Geometries.  Every geometry of the atomic backward with sampling_ratio > 0: any pooled size and C, 1..8 levels with
 *     extension and level mapping, v0 / v1.  sampling_ratio <= 0 (adaptive grid: the term count depends on the RoI sizes)
 *     returns RSDET_EINVAL and its workspace query returns 0.
 *   Limit.  K * pooled_h * pooled_w * sampling_ratio^2 * 4 <= 2^28 terms and batch * sum_l(H_l * W_l) < 2^32 - 1 pixels;
 *     above either RSDET_ELIMIT (the workspace query returns 0).
 *   Resources.  No atomics, no host synchronisation, no allocation: every scratch buffer, the radix sort's temporary
 *     storage included, comes from the workspace, whose query is host-only.  Safe under CUDA-graph capture. */
size_t rsdet_roi_align_rotated_backward_deterministic_workspace_bytes(const rsdet_roi_align_cfg* cfg, int num_rois,
                                                                      int feat_dtype);
int rsdet_roi_align_rotated_backward_deterministic(const rsdet_roi_align_cfg* cfg, int grad_out_dtype, const void* grad_out,
                                                   const float* rois, int num_rois, int feat_dtype, void* const* grad_feats_host,
                                                   void* workspace, size_t workspace_bytes, void* stream);

/* Measurement aid (bench.py's roofline): arm two cudaEvent_t (created with timing enabled by the caller).  The NEXT
 * rsdet_roi_align_rotated_forward call issued by this host thread records `start_event` right before and `stop_event`
 * right after its gather kernel on the call's stream (the geometry / order / transpose kernels of the call stay outside),
 * then disarms.  Pass NULLs to disarm.  No reference counterpart. */
int rsdet_roi_align_profile_events(void* start_event, void* stop_event);

/* NCHW <-> NHWC transposes of one fp32 map (exposed so a caller can keep a channels-last pyramid). */
int rsdet_nchw_to_nhwc(const float* src, int n, int c, int h, int w, float* dst, void* stream);
int rsdet_nhwc_to_nchw(const float* src, int n, int c, int h, int w, float* dst, void* stream);

/* ops/nms_poly.py:247-252 `iou_poly` (Shapely in the reference; convex clipping in float64 here) for n
 * ALIGNED pairs: polys1 (n,8), polys2 (n,8) fp64 -> ious (n) fp64 = inter / max(a1 + a2 - inter, 0.01). */
int rsdet_iou_poly_pairs(const double* polys1, const double* polys2, int n, double* ious, void* stream);

/* ---------------------------------------------------------------- merge-stage helper
 * data/devkits/result_merge.py:196-203 poly2origpoly: scene = (tile_poly + (x,y)) / rate, fp64.
 * polys (n,8) fp64 in-tile coords; offs (n,3) fp64 [x, y, rate] per row. */
int rsdet_poly2origpoly(const double* polys, const double* offs, int n, double* out, void* stream);

/* ---------------------------------------------------------------- SURVEY 8(f) rank 1: head tail fusion
 * models/roi_heads/oriented_head.py:498-536 (get_bboxes) + :279-305 (get_results), with
 * OrientedDeltaXYWHTCoder.decode (models/boxes/coder.py:477-514), regular_theta / regular_obb
 * (ops/bbox_transforms.py:501-519) and obb2poly (:612-623): softmax over (k, C+1) logits (background =
 * LAST column), delta decode against rois5 (k,5) [cx,cy,w,h,theta], optional division of cx,cy,w,h by
 * scale_factor4_host (NULL = rescale False), `score > score_thresh`, polygon conversion and compaction
 * in row-major (roi, class) order.  bbox_pred is (k,5) when reg_class_agnostic else (k,5*C).
 * means5_host / stds5_host / scale_factor4_host are HOST arrays (config constants).
 * out_dets (k*C, 9) [x1..y4, score], out_labels int64 (k*C), out_count int32 (1, device). */
size_t rsdet_oriented_head_results_workspace_bytes(int k);
int rsdet_oriented_head_results(const float* rois5, const float* cls_score, const float* bbox_pred, int k, int num_classes,
                                int reg_class_agnostic, const float* means5_host, const float* stds5_host, float wh_ratio_clip,
                                const float* scale_factor4_host, float score_thresh, int apply_softmax, float* out_dets,
                                int64_t* out_labels, int32_t* out_count, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- SURVEY 8(f) rank 3: evaluation matching
 * data/devkits/voc_eval.py:236-318 (voc_eval_dota), one class: detections (nd,8) fp64 polygons ALREADY in
 * descending-confidence order with their image index det_img (nd); ground truths (num_gts,8) grouped by
 * image (gt_start[num_imgs+1]), gt_difficult uint8 (num_gts).  Per detection: hbb prefilter (the reference's
 * +1 convention), iou_poly on the survivors, first maximum -> ovmax (nd, -inf if none), jmax (nd, global gt
 * index or -1); then the TP/FP marking of :303-311 (a gt is claimed by its highest-confidence match):
 * tp, fp uint8 (nd).  claim: int32 (num_gts) scratch. */
int rsdet_voc_match(const double* det_polys, const int32_t* det_img, int nd, const double* gt_polys, const int32_t* gt_start,
                    const uint8_t* gt_difficult, int num_imgs, int num_gts, double ovthresh, double* ovmax, int32_t* jmax,
                    int32_t* claim, uint8_t* tp, uint8_t* fp, void* stream);

/* ---------------------------------------------------------------- SURVEY 8(f) rank 2: oriented RPN proposals
 * models/roi_heads/oriented_rpn_head.py:136-216 (_get_bboxes_single), one image: per level sigmoid (or 2-way
 * softmax) of the (A*c, H, W) class map read in (h, w, a) order, top `nms_pre` by score when the level has
 * more (:183-190), MidpointOffsetCoder.decode (models/boxes/coder.py:383-433 with rectpoly2obb / regular_obb
 * ops/bbox_transforms.py:577-599, 501-519), min_bbox_size filter (:200-206), obb2hbb + per-level coordinate
 * offset (:208-211), jt.nms at nms_thresh, first nms_post rows.
 *   cls_scores[l]  (A or 2A, H_l, W_l) fp32;  bbox_preds[l] (A*6, H_l, W_l) fp32;  anchors[l] (H_l*W_l*A, 4)
 *   fp32 [x1,y1,x2,y2] in (h, w, a) order;  all device pointers, the pointer arrays live on the host.
 *   dets (nms_post, 6) fp32 [cx,cy,w,h,theta,score] in descending score order, num_dets int32 (1).
 * Optional candidate dump for parity tests (NULL to skip), ncand = sum_l min(n_l, nms_pre) rows in level
 * order: cand_obb (ncand,5), cand_hbb (ncand,4) WITH the level offsets, cand_score (ncand) (-inf where the
 * size filter dropped the row), cand_level int32 (ncand). */
typedef struct rsdet_rpn_cfg {
    int num_levels;               /* <= 8 */
    int height[8], width[8];
    int num_anchors;              /* A per location */
    int use_sigmoid;              /* 1: A class channels; 0: 2A channels, foreground = softmax(...)[:,1] */
    int nms_pre, nms_post;
    double nms_thresh;
    float min_bbox_size;          /* < 0 disables the filter */
    float means[6], stds[6];
    float wh_ratio_clip;          /* 16/1000 */
} rsdet_rpn_cfg;
int rsdet_rpn_num_candidates(const rsdet_rpn_cfg* cfg);
size_t rsdet_rpn_proposals_workspace_bytes(const rsdet_rpn_cfg* cfg);
int rsdet_rpn_proposals(const rsdet_rpn_cfg* cfg, const float* const* cls_scores, const float* const* bbox_preds,
                        const float* const* anchors, float* dets, int32_t* num_dets, float* cand_obb, float* cand_hbb,
                        float* cand_score, int32_t* cand_level, void* workspace, size_t workspace_bytes, void* stream);

/* counters for bench.py's `gpu_launches`: number of kernels this library has launched so far */
unsigned long long rsdet_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* RSDET_H_ */
