#!/usr/bin/env python
"""Generate tests/golden/oracle_drift_golden.npz: the ORACLE's own output (oracle/rsdet_oracle.c) on the inputs of
tests/test_oracle_vs_ref.py and the per-class keep counts of tests/test_gpu_nms.py::test_multiclass_nms_rotated_baseline_sizes.

    python tests/golden/make_golden_oracle_drift.py

This is a DRIFT GUARD, not reference output (the same status as the `merge_*` entries of rotated_path_golden.npz): it
makes any change of the oracle's arithmetic on these inputs fail without the reference tree.  It does not show that the
oracle equals the reference; that is shown by the comparisons with oracle/_ref in the same tests (which need the
reference tree) and, on smaller inputs, by tests/test_golden.py against rotated_path_golden.npz (reference output).

Arrays larger than SAMPLE elements are stored as a fixed seeded sample with its flat indices (`<key>_idx`), drawn
separately from the nonzero elements (three quarters) and the zero elements (one quarter) so that mostly-zero IoU
matrices are still sampled where boxes overlap.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
import test_oracle_vs_ref as T  # noqa: E402
import workloads as W  # noqa: E402
from oracle import oracle as O  # noqa: E402

SAMPLE = 8192
g = {}


def put(key, a):
    a = np.asarray(a).ravel()
    if a.size <= SAMPLE:
        g[key] = a
        return
    rng = np.random.default_rng(0)
    nz, z = np.flatnonzero(a != 0), np.flatnonzero(a == 0)
    k_nz = min(nz.size, SAMPLE * 3 // 4)
    k_z = min(z.size, SAMPLE - k_nz)
    idx = np.sort(np.concatenate([rng.choice(nz, k_nz, replace=False), rng.choice(z, k_z, replace=False)]))
    g[key], g[key + "_idx"] = a[idx], idx.astype(np.int32)


O.build()
G, P = T._pairs()
for v in (0, 1):
    for cs in (0, 1):
        put(f"iou_v{v}_cudasort{cs}", O.box_iou_rotated(G, P, v, cs))
        g[f"iou_degenerate_v{v}_cudasort{cs}"] = O.box_iou_rotated(T.DEGENERATE, T.DEGENERATE, v, cs)
d, order = T.nms_inputs()
for thr in (0.1, 0.5):
    for ge in (0, 1):
        g[f"nms_keep_{thr}_ge{ge}"] = O.nms_rotated_keep(d, order, thr, 5, bool(ge))
d6, order6 = T.ml_nms_inputs()
g["ml_nms_keep_0.1"] = O.nms_rotated_keep(d6, order6, 0.1, 6, False)
for v in (0, 1):
    for sr in (2, 0):
        feat, rois, rng = T.roi_inputs()
        a = O.roi_align_rotated_fwd(feat, rois, (7, 7), 1 / 16, sr, v)
        grad = rng.standard_normal(a.shape).astype(np.float32)
        put(f"roi_fwd_v{v}_sr{sr}", a)
        put(f"roi_bwd_v{v}_sr{sr}", O.roi_align_rotated_bwd(grad, rois, feat.shape, 1 / 16, sr, v))
pp, q, far = T.poly_inputs()
put("poly_iou", O.poly_iou_matrix(pp, pp))
put("poly_iou_far_reversed", O.poly_iou_matrix(q, far))
b9, _ = T.poly_nms_inputs()
g["poly_nms_keep_0.1"] = O.poly_nms(b9, 0.1)
# per-class keep counts of the CUDA-rule NMS (`>`) on the bench tiles (test_multiclass_nms_rotated_baseline_sizes)
for K, C, score_thr in ((4000, 10, 0.001), (2000, 15, 0.05)):
    boxes = W.rotated_boxes(K, 500)
    scores = W.class_scores(K, C, 0, logit_scale=1.0)
    kept = []
    for c in range(C):
        m = scores[:, c + 1] > np.float32(score_thr)
        o = np.argsort(-scores[m, c + 1].astype(np.float64), kind="stable").astype(np.int32)
        kept.append(int(O.nms_rotated_keep(boxes[m], o, 0.1, 5, False).sum()))
    g[f"mcnms_class_kept_K{K}_C{C}"] = np.array(kept, np.int64)
out = os.path.join(HERE, "oracle_drift_golden.npz")
np.savez_compressed(out, **g)
print("wrote", out, os.path.getsize(out), "bytes;", len(g), "arrays")
