"""jdet.models.boxes.iou_calculator -- python/jdet/models/boxes/iou_calculator.py: the rotated calculators (:81-162) and
BboxOverlaps2D, the horizontal default of MaxIoUAssigner (mode='iou', not aligned only)."""
from .... import core
from ...ops._io import back, dev
from ...ops.box_iou_rotated import box_iou_rotated
from ...ops.box_iou_rotated_v1 import box_iou_rotated_v1


def bbox_overlaps_rotated(rboxes1, rboxes2, version=0):
    if version == 0:
        ious = box_iou_rotated(rboxes1.float(), rboxes2.float())
    else:
        ious = box_iou_rotated_v1(rboxes1.float(), rboxes2.float())
    return ious


class _Rotated2D:
    version = 0

    def __call__(self, bboxes1, bboxes2, mode='iou', is_aligned=False):
        assert bboxes1.size(-1) in [0, 5, 6]
        assert bboxes2.size(-1) in [0, 5, 6]
        if bboxes2.size(-1) == 6:
            bboxes2 = bboxes2[..., :5]
        if bboxes1.size(-1) == 6:
            bboxes1 = bboxes1[..., :5]
        assert mode == "iou" and is_aligned == False  # noqa: E712 (as in the reference)
        return bbox_overlaps_rotated(bboxes1, bboxes2, version=self.version)

    def __repr__(self):
        return self.__class__.__name__ + '()'


class BboxOverlaps2D_rotated(_Rotated2D):
    """2D Overlaps Calculator, counter-clockwise convention (iou_calculator.py:81-115)."""
    version = 0


class BboxOverlaps2D_rotated_v1(_Rotated2D):
    """2D Overlaps Calculator, Oriented R-CNN convention (iou_calculator.py:117-155)."""
    version = 1


def bbox_overlaps(bboxes1, bboxes2):
    """(n1,4) x (n2,4) [x1,y1,x2,y2] -> (n1,n2) IoU; the formula is in include/rsdet.h (not pinned by a fixture)."""
    b1, fl = dev(bboxes1)
    b2, _ = dev(bboxes2)
    return back(core.bbox_overlaps(b1.reshape(-1, 4), b2.reshape(-1, 4)), fl)


class BboxOverlaps2D:
    """2D Overlaps Calculator for horizontal boxes.  (n,4) or (n,5) inputs; a fifth (score) column is dropped."""

    def __call__(self, bboxes1, bboxes2, mode='iou', is_aligned=False):
        assert bboxes1.size(-1) in [0, 4, 5]
        assert bboxes2.size(-1) in [0, 4, 5]
        if bboxes2.size(-1) == 5:
            bboxes2 = bboxes2[..., :4]
        if bboxes1.size(-1) == 5:
            bboxes1 = bboxes1[..., :4]
        assert mode == "iou" and is_aligned == False  # noqa: E712 (as the rotated calculators)
        return bbox_overlaps(bboxes1, bboxes2)

    def __repr__(self):
        return self.__class__.__name__ + '()'
