"""CPU restatement of the horizontal IoU (BboxOverlaps2D) that the anchor-assignment tests compare against.

mode='iou', not aligned: the mmdet 2.x bbox_overlaps, which JDet's models/boxes/iou_calculator.py copies.  fp32, no
"+1", each operation rounded to float32 on its own.  Restated, not pinned by a reference fixture (DESIGN.md section 3).
The assignment itself is checked with oracle.max_iou_assign over this matrix."""
import numpy as np

_f = np.float32


def bbox_overlaps(bboxes1, bboxes2):
    """(n1,4) x (n2,4) [x1,y1,x2,y2] -> (n1,n2) float32."""
    a = np.asarray(bboxes1, np.float32).reshape(-1, 4)[:, None, :]
    b = np.asarray(bboxes2, np.float32).reshape(-1, 4)[None, :, :]
    area_a = (a[..., 2] - a[..., 0]) * (a[..., 3] - a[..., 1])
    area_b = (b[..., 2] - b[..., 0]) * (b[..., 3] - b[..., 1])
    w = np.maximum(np.minimum(a[..., 2], b[..., 2]) - np.maximum(a[..., 0], b[..., 0]), _f(0))
    h = np.maximum(np.minimum(a[..., 3], b[..., 3]) - np.maximum(a[..., 1], b[..., 1]), _f(0))
    overlap = w * h
    union = np.maximum((area_a + area_b) - overlap, _f(1e-6))
    return (overlap / union).astype(np.float32)
